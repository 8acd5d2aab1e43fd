"""GPU parity of the lookahead path (BASELINE configs[1]): x265cu_frame_init_lowres ->
x265cu_lowres_intra_batch -> x265cu_lookahead_cost_batch against the oracle restatement, which
test_lookahead_oracle_vs_ref.py pins to the real Lowres / LookaheadTLD / CostEstimateGroup classes."""
import numpy as np
import pytest

from common import load_oracle, pixel_dtype
from frame_helpers import gen_luma, MARGIN_X, MARGIN_Y, MVRANGE
from lookahead_helpers import OracleLookahead, full_plane, lowres_geometry, LOOKAHEAD_LAMBDA

pytestmark = pytest.mark.gpu
TRIPLES = [(0, 1, 1), (0, 2, 1), (0, 2, 2), (0, 3, 1), (0, 3, 2), (0, 3, 3), (1, 3, 2), (2, 3, 3)]


@pytest.fixture(scope="module")
def cu():
    import x265_b200
    return x265_b200.load()


def GpuLookahead(cu, frames, depth):
    """The product's host mirror (x265_b200/lookahead.py) with every frame initialised and intra-estimated."""
    from x265_b200.lookahead import Lookahead
    H, W = frames[0].shape
    la = Lookahead(cu, W, H, depth, len(frames))
    for i, img in enumerate(frames):
        la.init_frame(i, img)
    la.intra_batch(range(len(frames)))
    return la


@pytest.mark.parametrize("depth", [8, 10])
@pytest.mark.parametrize("size,noise", [((416, 240), False), ((200, 136), True), ((960, 544), False)])
def test_lookahead_gpu(cu, depth, size, noise):
    O = load_oracle(depth)
    W, H = size
    frames = [gen_luma(W, H, i, s1=17.0, s2=11.0, bits=depth, noise=noise) for i in range(4)]
    orc = OracleLookahead(O, frames, depth)
    gpu = GpuLookahead(cu, frames, depth)
    vw = orc.w8 * 8 + 2 * MARGIN_X
    for k in range(4):
        got = gpu.fr[1]["planes"][k].download(pixel_dtype(depth)).reshape(orc.fr[1]["planes"][k].shape)
        assert np.array_equal(got[:, :vw], orc.fr[1]["planes"][k][:, :vw]), "lowres plane %d" % k
    for i in range(4):
        assert np.array_equal(gpu.fr[i]["intraCost"].download(np.int32), orc.fr[i]["intraCost"])
        assert np.array_equal(gpu.fr[i]["intraMode"].download(np.uint8), orc.fr[i]["intraMode"])
        assert np.array_equal(gpu.fr[i]["lc0"].download(np.uint16), orc.fr[i]["lowresCosts"][(0, 0)])
        assert np.array_equal(gpu.fr[i]["rs0"].download(np.int32), orc.fr[i]["rowSatds"][(0, 0)])
        assert tuple(int(x) for x in gpu.fr[i]["out0"].download(np.int64)) == orc.fr[i]["costEst"][(0, 0)]
    for (p0, p1, b) in TRIPLES:
        a, c = gpu.cost(p0, p1, b), orc.cost(p0, p1, b)
        d0, d1 = b - p0, p1 - b
        r = gpu.fr[b]["res"][(d0, d1)]
        assert np.array_equal(gpu.fr[b]["mvs"][(0, d0)].download(np.int32).reshape(-1, 2), orc.fr[b]["mvs"][(0, d0)]), (p0, p1, b)
        assert np.array_equal(gpu.fr[b]["mvcosts"][(0, d0)].download(np.int32), orc.fr[b]["mvcosts"][(0, d0)])
        if p1 > b:
            assert np.array_equal(gpu.fr[b]["mvs"][(1, d1)].download(np.int32).reshape(-1, 2), orc.fr[b]["mvs"][(1, d1)])
        assert np.array_equal(r["lowresCosts"], orc.fr[b]["lowresCosts"][(d0, d1)]), (p0, p1, b)
        assert np.array_equal(r["rowSatds"], orc.fr[b]["rowSatds"][(d0, d1)])
        assert a == c and r["costEstAq"] == orc.fr[b]["costEst"][(d0, d1)][1], ((p0, p1, b), a, c)


@pytest.mark.parametrize("world", [2, 4])
def test_lookahead_frame_shards_equal_single(cu, world):
    """Lookahead frames sharded per rank (BASELINE configs[3], x265_b200/lookahead.py): `world` Lookahead instances emulate
    the ranks on one GPU -- each initialises only the frames it owns, receives the other frames' 4-plane blocks (the
    broadcast payload), estimates the triples whose b it owns.  All costs equal the single-instance run bit for bit."""
    from x265_b200.lookahead import Lookahead, owner, window_triples, conflict_free_batches
    depth, W, H, n = 8, 416, 240, 8
    frames = [gen_luma(W, H, i, s1=17.0, s2=11.0, bits=depth) for i in range(n)]
    triples = window_triples(n, 3)
    single = GpuLookahead(cu, frames, depth)
    want = {}
    for b in conflict_free_batches(triples):
        for t, c in zip(b, single.cost_batch(b)):
            want[t] = c
    ranks = [Lookahead(cu, W, H, depth, n) for _ in range(world)]
    for i in range(n):
        ranks[owner(i, world)].init_frame(i, frames[i])
    for i in range(n):                                   # "broadcast" of frame i's plane block from its owner
        src = ranks[owner(i, world)]
        payload = src.fr[i]["block"].download(np.uint8)
        assert np.array_equal(payload, single.fr[i]["block"].download(np.uint8))
        for r, la in enumerate(ranks):
            if r != owner(i, world):
                la.fr[i]["block"].upload(payload); la.planes_received(i)
    got = {}
    for r, la in enumerate(ranks):
        la.intra_batch([i for i in range(n) if owner(i, world) == r])
        mine = [t for t in triples if owner(t[2], world) == r]
        for b in conflict_free_batches(mine):
            for t, c in zip(b, la.cost_batch(b)):
                got[t] = c
    assert got == want
    for la in ranks:
        la.close()
    single.close()


@pytest.mark.parametrize("depth,lslices", [(8, 8), (10, 4)])
def test_lookahead_cooperative_slices_gpu(cu, depth, lslices):
    """estimateFrameCost with cooperative lookahead slices (presets medium / slow: 8 / 4; slicetype.cpp:3075-3112, 3143-3173):
    on the device every slice of a triple is its own wavefront job; costs, motion fields, per-CU costs and row sums equal the
    oracle's slice loop, which tests/test_lookahead_oracle_vs_ref.py pins to the real Lookahead."""
    from x265_b200.lookahead import Lookahead, coop_slices
    O = load_oracle(depth)
    W, H = 1280, 720
    frames = [gen_luma(W, H, i, bits=depth) for i in range(3)]
    sl = coop_slices(H, lslices)
    assert sl[0] > 1
    orc = OracleLookahead(O, frames, depth, slices=sl)
    la = Lookahead(cu, W, H, depth, len(frames), lookahead_slices=lslices)
    for i, img in enumerate(frames):
        la.init_frame(i, img)
    la.intra_batch(range(len(frames)))
    for (p0, p1, b) in [(0, 1, 1), (0, 2, 1), (0, 2, 2)]:
        a, c = la.cost(p0, p1, b), orc.cost(p0, p1, b)
        d0, d1 = b - p0, p1 - b
        r = la.fr[b]["res"][(d0, d1)]
        assert np.array_equal(la.fr[b]["mvs"][(0, d0)].download(np.int32).reshape(-1, 2), orc.fr[b]["mvs"][(0, d0)]), (p0, p1, b)
        assert np.array_equal(r["lowresCosts"], orc.fr[b]["lowresCosts"][(d0, d1)]), (p0, p1, b)
        assert np.array_equal(r["rowSatds"], orc.fr[b]["rowSatds"][(d0, d1)])
        assert a == c and r["costEstAq"] == orc.fr[b]["costEst"][(d0, d1)][1], ((p0, p1, b), a, c)
    la.close()


@pytest.mark.parametrize("depth,lslices", [(8, 8), (10, 0)])
def test_lookahead_adaptive_quant_gpu(cu, depth, lslices):
    """The lookahead as preset medium runs it: adaptive quantisation weights from the REAL calcAdaptiveQuantFrame
    (oracle/_ref, slicetype.cpp:444-694) uploaded as Lowres::invQscaleFactor; intra estimate and frame costs on the device
    (costEst, costEstAq, AQ-weighted row sums, with and without cooperative slices) equal the oracle, which
    tests/test_lookahead_oracle_vs_ref.py::test_lookahead_with_adaptive_quant pins to the reference."""
    from test_lookahead_oracle_vs_ref import aq_inputs, AQ_TRIPLES
    from x265_b200.lookahead import Lookahead, coop_slices
    O = load_oracle(depth)
    W, H = 1280, 720
    frames, invq, ref_costs = aq_inputs(depth, lslices)
    assert any((q != 256).any() for q in invq)
    sl = coop_slices(H, lslices)
    orc = OracleLookahead(O, frames, depth, slices=sl if sl[0] > 1 else None, invq=invq)
    la = Lookahead(cu, W, H, depth, len(frames), lookahead_slices=lslices)
    for i, img in enumerate(frames):
        la.init_frame(i, img)
        la.set_invqscale(i, invq[i])
    la.intra_batch(range(len(frames)))
    for i in range(3):
        assert np.array_equal(la.fr[i]["intraCost"].download(np.int32), orc.fr[i]["intraCost"])
        assert np.array_equal(la.fr[i]["rs0"].download(np.int32), orc.fr[i]["rowSatds"][(0, 0)])
        assert tuple(int(x) for x in la.fr[i]["out0"].download(np.int64)) == orc.fr[i]["costEst"][(0, 0)]
    for (p0, p1, b), ref_cost in zip(AQ_TRIPLES, ref_costs):
        a, c = la.cost(p0, p1, b), orc.cost(p0, p1, b)
        d0, d1 = b - p0, p1 - b
        r = la.fr[b]["res"][(d0, d1)]
        assert a == c == ref_cost, (p0, p1, b)
        assert r["costEstAq"] == orc.fr[b]["costEst"][(d0, d1)][1]
        assert np.array_equal(r["rowSatds"], orc.fr[b]["rowSatds"][(d0, d1)])
        assert np.array_equal(r["lowresCosts"], orc.fr[b]["lowresCosts"][(d0, d1)])
    la.close()
