"""Pins the oracle's frame-level CTU-analysis driver against the same driver running on the REAL
reference code (MotionEstimate class + C primitive table, oracle/_ref).  CPU only."""
import numpy as np
import pytest

from common import load_oracle, RefResults, same
from frame_helpers import Workload, cpu_analyse, lambda_for, MVRANGE
from me_helpers import mvcost_table


FIELDS = ("njobs", "ncu", "jobs", "me_out", "cu_jobs", "cus", "cu_ref", "coef", "cu_sse", "cu_numsig", "recon", "intra_cost")


def ref_analyse(rec, wl, tab):
    """The frame driver on the reference code: run live while recording, read back from the golden file otherwise."""
    out = cpu_analyse(rec.R, "x265ref_analyse_frame", wl, tab, threads=4) if rec.recording else {}
    return rec({k: out[k] for k in FIELDS if k in out})


def compare(a, b):
    assert a["njobs"] == b["njobs"] and a["ncu"] == b["ncu"]
    assert same(a["jobs"], b["jobs"])
    assert same(a["me_out"], b["me_out"])
    assert same(a["cu_jobs"], b["cu_jobs"]) and same(a["cus"], b["cus"])
    assert same(a["cu_ref"], b["cu_ref"])
    assert same(a["coef"], b["coef"])
    assert same(a["cu_sse"], b["cu_sse"]) and same(a["cu_numsig"], b["cu_numsig"])
    assert len(a["recon"]) == len(b["recon"])
    for x, y in zip(a["recon"], b["recon"]):
        assert same(x, y)
    assert same(a["intra_cost"], b["intra_cost"])


@pytest.mark.parametrize("depth", [8, 10])
@pytest.mark.parametrize("noise", [False, True])
def test_frame_driver(depth, noise):
    rec = RefResults("frame_driver_%d_%d" % (depth, int(noise)), depth)
    R = rec.R
    O = load_oracle(depth)
    qp = 30
    wl = Workload(200, 136, depth=depth, numRefs=2, method=3, subme=3, merange=57, rect=1, qp=qp, noise=noise)
    tab = mvcost_table(O, R.x265ref_lambda(qp))
    assert abs(float(rec(np.array([R.x265ref_lambda(qp)]))[0]) - lambda_for(qp, depth)) < 1e-9
    a = cpu_analyse(O, "orc_analyse_frame", wl, tab, threads=4)
    b = ref_analyse(rec, wl, tab)
    assert a["njobs"] > 2000 and a["cu_numsig"].sum() > 0
    compare(a, b)
    rec.done()


@pytest.mark.parametrize("depth", [8, 10])
@pytest.mark.parametrize("noise", [False, True])
def test_frame_driver_chroma(depth, noise):
    """The same frame with 4:2:0 chroma planes: every ME job runs as the encoder's setSourcePU(Yuv, ..., bChroma = true) call,
    i.e. with the chroma-SATD term of subpelCompare for the PUs that have one (motion.cpp:204-212, 1601-1661)."""
    rec = RefResults("frame_driver_chroma_%d_%d" % (depth, int(noise)), depth)
    R = rec.R
    O = load_oracle(depth)
    qp = 30
    wl = Workload(200, 136, depth=depth, numRefs=2, method=3, subme=3, merange=57, rect=1, qp=qp, noise=noise, chroma=True)
    tab = mvcost_table(O, R.x265ref_lambda(qp))
    a = cpu_analyse(O, "orc_analyse_frame", wl, tab, threads=4)
    b = ref_analyse(rec, wl, tab)
    compare(a, b)
    rec.done()
    # the term is really on: results differ from the luma-only run of the same frame
    wl.chroma = False
    c = cpu_analyse(O, "orc_analyse_frame", wl, tab, threads=4)
    assert np.array_equal(a["jobs"], c["jobs"])
    assert (a["me_out"][:, 0] != c["me_out"][:, 0]).mean() > 0.3


@pytest.mark.parametrize("depth", [8, 10])
def test_frame_driver_amp(depth):
    """rect + AMP partitions (presets slower / veryslow, BASELINE configs[3..4]): 2NxnU / 2NxnD / nLx2N / nRx2N of CUs >= 16."""
    rec = RefResults("frame_driver_amp_%d" % depth, depth)
    R = rec.R
    O = load_oracle(depth)
    qp = 30
    wl = Workload(200, 136, depth=depth, numRefs=2, method=3, subme=4, merange=57, rect=1, qp=qp, amp=1)
    tab = mvcost_table(O, R.x265ref_lambda(qp))
    a = cpu_analyse(O, "orc_analyse_frame", wl, tab, threads=4)
    b = ref_analyse(rec, wl, tab)
    sizes = {(int(j["pw"]), int(j["ph"])) for j in a["jobs"]}
    assert {(64, 16), (64, 48), (16, 64), (48, 64), (32, 8), (32, 24), (8, 32), (24, 32), (16, 4), (16, 12), (4, 16), (12, 16)} <= sizes
    compare(a, b)
    rec.done()
