"""Generates tests/golden/primitives_{8,10}.npz from the REAL reference (oracle/_ref/libx265ref*.so,
compiled from /root/reference by oracle/Makefile.ref).  Run in the build container only:
    python tests/golden/make_golden.py          (primitives_*.npz, me_chroma_*.npz)
    python tests/golden/make_golden.py --ref    (ref/*.npz, the results the *_oracle_vs_ref tests replay)
Each entry stores the inputs and the reference's outputs, so the checks need no reference at run time."""
import ctypes as C
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE)); sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from common import LUMA_PU, LUMA_CU, P, I, IP, load_ref, load_oracle, ref_fn, ptr, pixel_dtype  # noqa: E402
from me_helpers import run_both, run_both_chroma, CHROMA_CASES  # noqa: E402


def gen(depth):
    R = load_ref(depth)
    rng = np.random.default_rng(2650 + depth)
    mx = (1 << depth) - 1
    dt = pixel_dtype(depth)
    sse_t = C.c_uint32 if depth == 8 else C.c_uint64
    g = {}
    a = rng.integers(0, mx + 1, (64, 64)).astype(dt); b = rng.integers(0, mx + 1, (72, 96)).astype(dt)
    g["cmp_a"], g["cmp_b"] = a, b
    for pu in (1, 2, 4, 6, 8, 14, 17, 22):
        w, h = LUMA_PU[pu]
        g["sad_%d" % pu] = np.int64(ref_fn(R, "pu.sad", I, [P, IP, P, IP], pu)(ptr(a), 64, ptr(b, 5), 96))
        g["satd_%d" % pu] = np.int64(ref_fn(R, "pu.satd", I, [P, IP, P, IP], pu)(ptr(a), 64, ptr(b, 5), 96))
    for cu in range(5):
        g["sa8d_%d" % cu] = np.int64(ref_fn(R, "cu.sa8d", I, [P, IP, P, IP], cu)(ptr(a), 64, ptr(b, 5), 96))
        g["sse_%d" % cu] = np.uint64(ref_fn(R, "cu.sse_pp", sse_t, [P, IP, P, IP], cu)(ptr(a), 64, ptr(b, 5), 96))
        g["psy_%d" % cu] = np.int64(ref_fn(R, "cu.psy_cost_pp", I, [P, IP, P, IP], cu)(ptr(a), 64, ptr(b, 5), 96))
        g["var_%d" % cu] = np.uint64(ref_fn(R, "cu.var", C.c_uint64, [P, IP], cu)(ptr(a), 64))
    # interpolation, 16x16 luma, all variants
    src = rng.integers(0, mx + 1, (40, 64)).astype(dt); ssrc = rng.integers(-4096, 4096, (40, 64)).astype(np.int16)
    g["ip_src"], g["ip_ssrc"] = src, ssrc
    s0 = 8 * 64 + 8
    for ci in range(1, 4):
        for nm, short_in, short_out in (("luma_hpp", 0, 0), ("luma_vpp", 0, 0), ("luma_vps", 0, 1), ("luma_vsp", 1, 0), ("luma_vss", 1, 1)):
            d = np.zeros((16, 16), np.int16 if short_out else dt)
            ref_fn(R, "pu." + nm, None, [P, IP, P, IP, I], 2)(ptr(ssrc if short_in else src, s0), 64, ptr(d), 16, ci)
            g["%s_%d" % (nm, ci)] = d
        d = np.zeros((23, 16), np.int16)
        ref_fn(R, "pu.luma_hps", None, [P, IP, P, IP, I, I], 2)(ptr(src, s0), 64, ptr(d), 16, ci, 1)
        g["luma_hps_ext_%d" % ci] = d
        for cj in range(1, 4):
            d = np.zeros((16, 16), dt)
            ref_fn(R, "pu.luma_hvpp", None, [P, IP, P, IP, I, I], 2)(ptr(src, s0), 64, ptr(d), 16, ci, cj)
            g["luma_hvpp_%d%d" % (ci, cj)] = d
    # transforms / quant
    for cu, n in enumerate(LUMA_CU[:4]):
        res = (rng.integers(0, mx + 1, (n, n)) - rng.integers(0, mx + 1, (n, n))).astype(np.int16)
        g["tr_res_%d" % n] = res
        co = np.zeros(n * n, np.int16); ref_fn(R, "cu.dct", None, [P, P, IP], cu)(ptr(res), ptr(co), n); g["dct_%d" % n] = co
        back = np.zeros((n, n), np.int16); ref_fn(R, "cu.idct", None, [P, P, IP], cu)(ptr(co), ptr(back), n); g["idct_%d" % n] = back
        qc = np.full(n * n, 18396, np.int32); du = np.zeros(n * n, np.int32); q = np.zeros(n * n, np.int16)
        qbits = 14 + 5 + (15 - depth - (cu + 2)); add = 85 << (qbits - 9)
        ns = ref_fn(R, "quant", C.c_uint32, [P, P, P, P, I, I, I])(ptr(co), ptr(qc), ptr(du), ptr(q), qbits, add, n * n)
        g["quant_%d" % n], g["quant_du_%d" % n], g["quant_ns_%d" % n], g["quant_par_%d" % n] = q, du, np.int64(ns), np.array([qbits, add])
        dq = np.zeros(n * n, np.int16); ref_fn(R, "dequant_normal", None, [P, P, I, I, I])(ptr(q), ptr(dq), n * n, 57 << 5, 6 - (15 - depth - (cu + 2))); g["dequant_%d" % n] = dq
    res4 = g["tr_res_4"]; co = np.zeros(16, np.int16); ref_fn(R, "dst4x4", None, [P, P, IP])(ptr(res4), ptr(co), 4); g["dst4"] = co
    # intra
    for cu, n in enumerate(LUMA_CU[:4]):
        nb = rng.integers(0, mx + 1, 4 * n + 1).astype(dt); g["intra_nb_%d" % n] = nb
        f = np.zeros(4 * n + 1, dt); ref_fn(R, "cu.intra_filter", None, [P, P], cu)(ptr(nb), ptr(f)); g["intra_filt_%d" % n] = f
        out = np.zeros((35, n, n), dt)
        for m in range(35):
            ref_fn(R, "cu.intra_pred", None, [P, IP, P, I, I], cu, m)(ptr(out[m]), n, ptr(nb), m, 1 if n <= 16 else 0)
        g["intra_pred_%d" % n] = out
    # motion estimation: results of the real MotionEstimate on seeded planes (inputs are regenerated from the seed)
    O = load_oracle(depth)
    me = []
    mrng = np.random.default_rng(77 + depth)
    for method in (0, 1, 3):
        for (w, h) in ((8, 8), (16, 16), (32, 16), (64, 64), (8, 4)):
            for subme in (1, 3, 5):
                r, o = run_both(O, R, depth, mrng, w, h, method, subme, 0, True, 57 if method == 3 else 16)
                assert r == o
                me.append([method, w, h, subme] + list(r))
    g["me_results"] = np.array(me, np.int64)
    np.savez_compressed(os.path.join(HERE, "primitives_%d.npz" % depth), **g)
    print("wrote primitives_%d.npz with %d arrays" % (depth, len(g)))


def gen_chroma(depth):
    """4:2:0 motionEstimate with the chroma-SATD term (motion.cpp:1601-1661): results of the real MotionEstimate driven
    through the Yuv variant of setSourcePU (x265ref_motion_estimate_chroma); inputs are regenerated from the seed."""
    R = load_ref(depth)
    O = load_oracle(depth)
    rng = np.random.default_rng(177 + depth)
    rows = []
    for (method, w, h, subme) in CHROMA_CASES:
        r, o = run_both_chroma(O, R, depth, rng, w, h, method, subme, True, 57 if method == 3 else 16)
        assert r == o
        rows.append([method, w, h, subme] + list(r))
    np.savez_compressed(os.path.join(HERE, "me_chroma_%d.npz" % depth), me_results=np.array(rows, np.int64))
    print("wrote me_chroma_%d.npz with %d jobs" % (depth, len(rows)))


# the tests that replay the reference's results from tests/golden/ref (common.RefResults)
REF_TESTS = ["tests/test_oracle_vs_ref.py", "tests/test_frame_oracle_vs_ref.py", "tests/test_lookahead_oracle_vs_ref.py"]


def gen_ref_results():
    """Rewrites tests/golden/ref/*.npz: the tests run with the reference live and record what it computed."""
    import subprocess
    root = os.path.dirname(os.path.dirname(HERE))
    env = dict(os.environ, X265_RECORD_GOLDEN="1")
    subprocess.check_call([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider"] + REF_TESTS, cwd=root, env=env)


if __name__ == "__main__":
    if "--ref" in sys.argv:
        gen_ref_results()
        sys.exit(0)
    for d in (8, 10):
        if "--chroma-only" not in sys.argv:
            gen(d)
        gen_chroma(d)
