"""Table-vs-oracle checks shared by the CPU pin (reference C table vs oracle, test_oracle_vs_ref.py)
and the GPU parity tests (CUDA per-call table vs oracle, test_gpu_table.py).

`get(name, restype, argtypes, i, j, k)` returns a callable for an EncoderPrimitives field or None; `ref_out` maps each output
array of the table under test to what is compared (a RefResults substitutes the reference's stored outputs).
Mirrors the reference TestBench (source/test/testbench.cpp:155-233): same inputs through both
tables, exact equality, fixtures random / all-min / all-max.
"""
import ctypes as C
import numpy as np

from common import (LUMA_PU, LUMA_CU, CSP_I420, P, I, IP, ptr, fixtures, resid_fixture, pixel_dtype, same)

def check_pixelcmp(get, O, depth, kind, ref_out=lambda v: v):
    rng = np.random.default_rng(1)
    for pu, (w, h) in enumerate(LUMA_PU):
        a = fixtures(rng, depth, (64 + 8, 64), kind)
        b = fixtures(rng, depth, (64 + 8, 200), "rand" if kind == "rand" else ("max" if kind == "min" else "min"))
        for name, ofn in (("pu.sad", O.orc_sad), ("pu.satd", O.orc_satd)):
            f = get(name, I, [P, IP, P, IP], pu)
            assert f(ptr(a), 64, ptr(b, 3), 200) == ofn(ptr(a), IP(64), ptr(b, 3), IP(200), w, h), (name, w, h)
        # sad_x3 / x4
        res_r = np.zeros(4, np.int32); res_o = np.zeros(4, np.int32)
        f4 = get("pu.sad_x4", None, [P, P, P, P, P, IP, P], pu)
        f4(ptr(a), ptr(b, 0), ptr(b, 5), ptr(b, 200), ptr(b, 407), 200, ptr(res_r))
        O.orc_sad_x4(ptr(a), ptr(b, 0), ptr(b, 5), ptr(b, 200), ptr(b, 407), IP(200), ptr(res_o), w, h)
        assert same(ref_out(res_r), res_o)
        f3 = get("pu.sad_x3", None, [P, P, P, P, IP, P], pu)
        res_r[:] = 0; res_o[:] = 0
        f3(ptr(a), ptr(b, 1), ptr(b, 7), ptr(b, 201), 200, ptr(res_r))
        O.orc_sad_x3(ptr(a), ptr(b, 1), ptr(b, 7), ptr(b, 201), IP(200), ptr(res_o), w, h)
        assert same(ref_out(res_r), res_o)
    for cu, n in enumerate(LUMA_CU):
        a = fixtures(rng, depth, (64, 64), kind)
        b = fixtures(rng, depth, (64, 96), "rand" if kind == "rand" else ("max" if kind == "min" else "min"))
        f = get("cu.sa8d", I, [P, IP, P, IP], cu)
        assert f(ptr(a), 64, ptr(b), 96) == O.orc_sa8d(ptr(a), IP(64), ptr(b), IP(96), n, n), ("sa8d", n)
        sse = C.c_uint32 if depth == 8 else C.c_uint64
        f = get("cu.sse_pp", sse, [P, IP, P, IP], cu)
        assert f(ptr(a), 64, ptr(b), 96) == O.orc_sse_pp(ptr(a), IP(64), ptr(b), IP(96), n, n)
        f = get("cu.psy_cost_pp", I, [P, IP, P, IP], cu)
        assert f(ptr(a), 64, ptr(b), 96) == O.orc_psy_cost_pp(ptr(a), IP(64), ptr(b), IP(96), n)
        f = get("cu.var", C.c_uint64, [P, IP], cu)
        assert f(ptr(a), 64) == O.orc_var(ptr(a), IP(64), n)
        sa = resid_fixture(rng, depth, (64, 64), kind); sb = resid_fixture(rng, depth, (64, 64), "rand")
        f = get("cu.sse_ss", sse, [P, IP, P, IP], cu)
        assert f(ptr(sa), 64, ptr(sb), 64) == O.orc_sse_ss(ptr(sa), IP(64), ptr(sb), IP(64), n, n)
        f = get("cu.ssd_s", sse, [P, IP], cu, 0)
        assert f(ptr(sa), 64) == O.orc_ssd_s(ptr(sa), IP(64), n)
    # 4:2:0 chroma aliases (primitives.cpp:88-209): chroma sa8d/satd of the chroma-sized block
    for pu, (w, h) in enumerate(LUMA_PU):
        cw, ch = w // 2, h // 2
        f = get("chroma.pu.satd", I, [P, IP, P, IP], pu, 0, CSP_I420)
        if f is None:
            assert cw % 4 or ch % 4
            continue
        a = fixtures(rng, depth, (64, 64), kind); b = fixtures(rng, depth, (64, 64), "rand")
        assert f(ptr(a), 64, ptr(b), 64) == O.orc_satd(ptr(a), IP(64), ptr(b), IP(64), cw, ch), ("chroma satd", w, h)
    for cu, n in enumerate(LUMA_CU):
        f = get("chroma.cu.sa8d", I, [P, IP, P, IP], cu, 0, CSP_I420)
        if f is None or n < 8:
            continue
        a = fixtures(rng, depth, (64, 64), kind); b = fixtures(rng, depth, (64, 64), "rand")
        assert f(ptr(a), 64, ptr(b), 64) == O.orc_sa8d(ptr(a), IP(64), ptr(b), IP(64), n // 2, n // 2), ("chroma sa8d", n)


def check_ads(get, O, depth, ref_out=lambda v: v):
    # not covered by the reference TestBench (SURVEY 4); checked directly against pixel.cpp:121-165
    rng = np.random.default_rng(2)
    for pu, (w, h) in enumerate(LUMA_PU):
        enc = rng.integers(0, 1 << 18, 4).astype(np.int32)
        sums = rng.integers(0, 1 << 18, 512).astype(np.uint32)
        cost = rng.integers(0, 2000, 256).astype(np.uint16)
        mr = np.zeros(256, np.int16); mo = np.zeros(256, np.int16)
        f = get("pu.ads", I, [P, P, I, P, P, I, I], pu)
        thresh = 1 << 17
        nr = f(ptr(enc), ptr(sums), 100, ptr(cost), ptr(mr), 116, thresh)
        no = O.orc_ads(ptr(enc), ptr(sums), 100, ptr(cost), ptr(mo), 116, thresh, w, h)
        assert nr == no and same(ref_out(mr[:nr]), mo[:no]), (w, h)


def check_blockops(get, O, depth, kind, ref_out=lambda v: v):
    rng = np.random.default_rng(3)
    dt = pixel_dtype(depth)
    for pu, (w, h) in enumerate(LUMA_PU):
        a = fixtures(rng, depth, (64, 80), kind); b = fixtures(rng, depth, (64, 72), "rand")
        dr = np.zeros((64, 96), dt); do = np.zeros((64, 96), dt)
        get("pu.pixelavg_pp", None, [P, IP, P, IP, P, IP, I], pu, 0)(ptr(dr), 96, ptr(a), 80, ptr(b), 72, 32)
        O.orc_pixelavg_pp(ptr(do), IP(96), ptr(a), IP(80), ptr(b), IP(72), w, h)
        assert same(ref_out(dr), do)
        dr[:] = 0; do[:] = 0
        get("pu.copy_pp", None, [P, IP, P, IP], pu)(ptr(dr), 96, ptr(a), 80)
        O.orc_copy_pp(ptr(do), IP(96), ptr(a), IP(80), w, h)
        assert same(ref_out(dr), do)
        s0 = rng.integers(-(1 << 13), 1 << 13, (64, 64)).astype(np.int16)
        s1 = rng.integers(-(1 << 13), 1 << 13, (64, 64)).astype(np.int16)
        if kind == "max":
            s0[:] = 32767; s1[:] = 32767
        if kind == "min":
            s0[:] = -32768; s1[:] = -32768
        dr[:] = 0; do[:] = 0
        get("pu.addAvg", None, [P, P, P, IP, IP, IP], pu, 0)(ptr(s0), ptr(s1), ptr(dr), 64, 64, 96)
        O.orc_addAvg(ptr(s0), ptr(s1), ptr(do), IP(64), IP(64), IP(96), w, h)
        assert same(ref_out(dr), do)
        sr = np.zeros((64, 64), np.int16); so = np.zeros((64, 64), np.int16)
        get("pu.convert_p2s", None, [P, IP, P, IP], pu, 0)(ptr(a), 80, ptr(sr), 64)
        O.orc_p2s(ptr(a), IP(80), ptr(so), IP(64), w, h)
        assert same(ref_out(sr), so)
    for cu, n in enumerate(LUMA_CU):
        a = fixtures(rng, depth, (64, 64), kind); b = fixtures(rng, depth, (64, 64), "rand")
        r = resid_fixture(rng, depth, (64, 64), kind)
        sr = np.zeros((64, 64), np.int16); so = np.zeros((64, 64), np.int16)
        get("cu.sub_ps", None, [P, IP, P, P, IP, IP], cu)(ptr(sr), 64, ptr(a), ptr(b), 64, 64)
        O.orc_sub_ps(ptr(so), IP(64), ptr(a), ptr(b), IP(64), IP(64), n, n)
        assert same(ref_out(sr), so)
        sr[:] = 0; so[:] = 0
        get("cu.calcresidual", None, [P, P, P, IP], cu, 0)(ptr(a), ptr(b), ptr(sr), 64)
        O.orc_calcresidual(ptr(a), ptr(b), ptr(so), IP(64), n)
        assert same(ref_out(sr), so)
        dr = np.zeros((64, 64), dt); do = np.zeros((64, 64), dt)
        get("cu.add_ps", None, [P, IP, P, P, IP, IP], cu, 0)(ptr(dr), 64, ptr(a), ptr(r), 64, 64)
        O.orc_add_ps(ptr(do), IP(64), ptr(a), ptr(r), IP(64), IP(64), n, n)
        assert same(ref_out(dr), do)
        dr[:] = 0; do[:] = 0
        get("cu.transpose", None, [P, P, IP], cu)(ptr(dr), ptr(a), 64)
        O.orc_transpose(ptr(do), ptr(a), IP(64), n)
        assert same(ref_out(dr), do)
        for nm, of in (("cu.copy_ss", O.orc_copy_ss),):
            sr[:] = 0; so[:] = 0
            get(nm, None, [P, IP, P, IP], cu)(ptr(sr), 64, ptr(r), 64)
            of(ptr(so), IP(64), ptr(r), IP(64), n, n)
            assert same(ref_out(sr), so)
        sr[:] = 0; so[:] = 0
        get("cu.copy_ps", None, [P, IP, P, IP], cu)(ptr(sr), 64, ptr(a), 64)
        O.orc_copy_ps(ptr(so), IP(64), ptr(a), IP(64), n, n)
        assert same(ref_out(sr), so)
        pos = np.abs(r) & ((1 << depth) - 1)
        dr[:] = 0; do[:] = 0
        get("cu.copy_sp", None, [P, IP, P, IP], cu)(ptr(dr), 64, ptr(pos), 64)
        O.orc_copy_sp(ptr(do), IP(64), ptr(pos), IP(64), n, n)
        assert same(ref_out(dr), do)
        if n <= 32:
            for shift in (1, 3):
                for nm, of, two_d_dst in (("cu.cpy2Dto1D_shl", O.orc_cpy2Dto1D_shl, False), ("cu.cpy2Dto1D_shr", O.orc_cpy2Dto1D_shr, False),
                                          ("cu.cpy1Dto2D_shl", O.orc_cpy1Dto2D_shl, True), ("cu.cpy1Dto2D_shr", O.orc_cpy1Dto2D_shr, True)):
                    sr[:] = 0; so[:] = 0
                    j = 0
                    get(nm, None, [P, P, IP, I], cu, j)(ptr(sr), ptr(r), 64, shift)
                    of(ptr(so), ptr(r), IP(64), shift, n)
                    assert same(ref_out(sr), so), nm
            sr[:] = 0; so[:] = 0
            nr = get("cu.copy_cnt", C.c_uint32, [P, P, IP], cu)(ptr(sr), ptr(r), 64)
            no = O.orc_copy_cnt(ptr(so), ptr(r), IP(64), n)
            assert nr == no and same(ref_out(sr), so)
            assert get("cu.count_nonzero", I, [P], cu)(ptr(r)) == O.orc_count_nonzero(ptr(r), n)
        sr[:] = 0; so[:] = 0
        get("cu.blockfill_s", None, [P, IP, C.c_int16], cu, 0)(ptr(sr), 64, -1234)
        O.orc_blockfill_s(ptr(so), IP(64), C.c_int16(-1234), n)
        assert same(ref_out(sr), so)
    # scale2D, lowres, weight
    a = fixtures(rng, depth, (66, 80), kind)
    dr = np.zeros(32 * 32, dt); do = np.zeros(32 * 32, dt)
    get("scale2D_64to32", None, [P, P, IP])(ptr(dr), ptr(a), 80)
    O.orc_scale2D_64to32(ptr(do), ptr(a), IP(80))
    assert same(ref_out(dr), do)
    src = fixtures(rng, depth, (130, 200), kind)
    outs_r = [np.zeros((64, 100), dt) for _ in range(4)]; outs_o = [np.zeros((64, 100), dt) for _ in range(4)]
    get("frameInitLowres", None, [P, P, P, P, P, IP, IP, I, I])(ptr(src), *[ptr(x) for x in outs_r], 200, 100, 96, 64)
    O.orc_frame_init_lowres(ptr(src), *[ptr(x) for x in outs_o], IP(200), IP(100), 96, 64)
    for x, y in zip(outs_r, outs_o):
        assert same(ref_out(x), y)
    a = fixtures(rng, depth, (32, 64), kind)
    dr = np.zeros((32, 64), dt); do = np.zeros((32, 64), dt)
    corr = 14 - depth
    get("weight_pp", None, [P, P, IP, I, I, I, I, I, I])(ptr(a), ptr(dr), 64, 48, 30, 70, 1 << (corr + 5), corr + 6, 3)
    O.orc_weight_pp(ptr(a), ptr(do), IP(64), 48, 30, 70, 1 << (corr + 5), corr + 6, 3)
    assert same(ref_out(dr), do)
    s = rng.integers(-8192, 8191, (32, 64)).astype(np.int16)
    dr[:] = 0; do[:] = 0
    get("weight_sp", None, [P, P, IP, IP, I, I, I, I, I, I])(ptr(s), ptr(dr), 64, 64, 47, 30, 70, 1 << (corr + 5), corr + 6, 3)
    O.orc_weight_sp(ptr(s), ptr(do), IP(64), IP(64), 47, 30, 70, 1 << (corr + 5), corr + 6, 3)
    assert same(ref_out(dr), do)


def check_interp(get, O, depth, kind, ref_out=lambda v: v):
    rng = np.random.default_rng(4)
    dt = pixel_dtype(depth)
    for pu, (w, h) in enumerate(LUMA_PU):
        src = fixtures(rng, depth, (64 + 16, 160), kind)
        ss = 160
        s0 = 8 * ss + 8
        ssrc = rng.integers(-(1 << 12), 1 << 12, (64 + 16, 160)).astype(np.int16)
        if kind == "max":
            ssrc[:] = 16383
        if kind == "min":
            ssrc[:] = -16384
        for ci in range(4):
            dr = np.zeros((64 + 8, 100), dt); do = np.zeros((64 + 8, 100), dt)
            for nm, of in (("pu.luma_hpp", O.orc_interp_hpp), ("pu.luma_vpp", O.orc_interp_vpp)):
                dr[:] = 0; do[:] = 0
                get(nm, None, [P, IP, P, IP, I], pu)(ptr(src, s0), ss, ptr(dr), 100, ci)
                of(ptr(src, s0), IP(ss), ptr(do), IP(100), ci, 8, w, h)
                assert same(ref_out(dr), do), (nm, w, h, ci)
            sr = np.zeros((64 + 8, 100), np.int16); so = np.zeros((64 + 8, 100), np.int16)
            for ext in (0, 1):
                sr[:] = 0; so[:] = 0
                get("pu.luma_hps", None, [P, IP, P, IP, I, I], pu)(ptr(src, s0), ss, ptr(sr), 100, ci, ext)
                O.orc_interp_hps(ptr(src, s0), IP(ss), ptr(so), IP(100), ci, ext, 8, w, h)
                assert same(ref_out(sr), so), ("hps", w, h, ci, ext)
            sr[:] = 0; so[:] = 0
            get("pu.luma_vps", None, [P, IP, P, IP, I], pu)(ptr(src, s0), ss, ptr(sr), 100, ci)
            O.orc_interp_vps(ptr(src, s0), IP(ss), ptr(so), IP(100), ci, 8, w, h)
            assert same(ref_out(sr), so)
            dr[:] = 0; do[:] = 0
            get("pu.luma_vsp", None, [P, IP, P, IP, I], pu)(ptr(ssrc, s0), ss, ptr(dr), 100, ci)
            O.orc_interp_vsp(ptr(ssrc, s0), IP(ss), ptr(do), IP(100), ci, 8, w, h)
            assert same(ref_out(dr), do)
            sr[:] = 0; so[:] = 0
            get("pu.luma_vss", None, [P, IP, P, IP, I], pu)(ptr(ssrc, s0), ss, ptr(sr), 100, ci)
            O.orc_interp_vss(ptr(ssrc, s0), IP(ss), ptr(so), IP(100), ci, 8, w, h)
            assert same(ref_out(sr), so)
            for cj in range(1, 4):
                if ci == 0:
                    continue
                dr[:] = 0; do[:] = 0
                get("pu.luma_hvpp", None, [P, IP, P, IP, I, I], pu)(ptr(src, s0), ss, ptr(dr), 100, ci, cj)
                O.orc_interp_hvpp(ptr(src, s0), IP(ss), ptr(do), IP(100), ci, cj, 8, w, h)
                assert same(ref_out(dr), do)
        # 4:2:0 chroma, 4-tap, block = (w/2, h/2)
        cw, ch = w // 2, h // 2
        for ci in (0, 1, 4, 7):
            dr = np.zeros((40, 100), dt); do = np.zeros((40, 100), dt)
            for nm, of in (("chroma.pu.filter_hpp", O.orc_interp_hpp), ("chroma.pu.filter_vpp", O.orc_interp_vpp)):
                f = get(nm, None, [P, IP, P, IP, I], pu, 0, CSP_I420)
                if f is None:
                    continue
                dr[:] = 0; do[:] = 0
                f(ptr(src, s0), ss, ptr(dr), 100, ci)
                of(ptr(src, s0), IP(ss), ptr(do), IP(100), ci, 4, cw, ch)
                assert same(ref_out(dr), do), (nm, w, h, ci)
            sr = np.zeros((40, 100), np.int16); so = np.zeros((40, 100), np.int16)
            f = get("chroma.pu.filter_hps", None, [P, IP, P, IP, I, I], pu, 0, CSP_I420)
            if f is not None:
                for ext in (0, 1):
                    sr[:] = 0; so[:] = 0
                    f(ptr(src, s0), ss, ptr(sr), 100, ci, ext)
                    O.orc_interp_hps(ptr(src, s0), IP(ss), ptr(so), IP(100), ci, ext, 4, cw, ch)
                    assert same(ref_out(sr), so)
            f = get("chroma.pu.filter_vps", None, [P, IP, P, IP, I], pu, 0, CSP_I420)
            if f is not None:
                sr[:] = 0; so[:] = 0
                f(ptr(src, s0), ss, ptr(sr), 100, ci)
                O.orc_interp_vps(ptr(src, s0), IP(ss), ptr(so), IP(100), ci, 4, cw, ch)
                assert same(ref_out(sr), so)
            f = get("chroma.pu.filter_vsp", None, [P, IP, P, IP, I], pu, 0, CSP_I420)
            if f is not None:
                dr[:] = 0; do[:] = 0
                f(ptr(ssrc, s0), ss, ptr(dr), 100, ci)
                O.orc_interp_vsp(ptr(ssrc, s0), IP(ss), ptr(do), IP(100), ci, 4, cw, ch)
                assert same(ref_out(dr), do)
            f = get("chroma.pu.filter_vss", None, [P, IP, P, IP, I], pu, 0, CSP_I420)
            if f is not None:
                sr[:] = 0; so[:] = 0
                f(ptr(ssrc, s0), ss, ptr(sr), 100, ci)
                O.orc_interp_vss(ptr(ssrc, s0), IP(ss), ptr(so), IP(100), ci, 4, cw, ch)
                assert same(ref_out(sr), so)


def check_transforms(get, O, depth, kind, ref_out=lambda v: v):
    rng = np.random.default_rng(5)
    for cu, n in enumerate(LUMA_CU[:4]):
        for it in range(8):
            src = resid_fixture(rng, depth, (32, 40), kind)
            if kind != "rand" and it % 2:
                src = -src
            dr = np.zeros(n * n, np.int16); do = np.zeros(n * n, np.int16)
            get("cu.dct", None, [P, P, IP], cu)(ptr(src), ptr(dr), 40)
            O.orc_dct(ptr(src), ptr(do), IP(40), n)
            assert same(ref_out(dr), do), ("dct", n)
            coef = rng.integers(-32768, 32768, n * n).astype(np.int16) if it < 4 else do.copy()     # == dr, checked above
            if kind == "max":
                coef[:] = 32767
            if kind == "min":
                coef[:] = -32768
            ir = np.zeros((32, 40), np.int16); io = np.zeros((32, 40), np.int16)
            get("cu.idct", None, [P, P, IP], cu)(ptr(coef), ptr(ir), 40)
            O.orc_idct(ptr(coef), ptr(io), IP(40), n)
            assert same(ref_out(ir), io), ("idct", n)
            if n == 4:
                get("dst4x4", None, [P, P, IP])(ptr(src), ptr(dr), 40)
                O.orc_dst4(ptr(src), ptr(do), IP(40))
                assert same(ref_out(dr), do)
                ir[:] = 0; io[:] = 0
                get("idst4x4", None, [P, P, IP])(ptr(coef), ptr(ir), 40)
                O.orc_idst4(ptr(coef), ptr(io), IP(40))
                assert same(ref_out(ir), io)
        # quant family (mbdstharness.cpp:139-300 style parameters)
        num = n * n
        for it in range(8):
            coef = rng.integers(-32768, 32768, num).astype(np.int16)
            if kind == "max":
                coef[:] = 32767
            if kind == "min":
                coef[:] = -32768
            qc = rng.integers(1, 1 << 16, num).astype(np.int32)
            qbits = int(rng.integers(8, 24)); add = int(rng.integers(0, 1 << (qbits - 1)))
            dur = np.zeros(num, np.int32); duo = np.zeros(num, np.int32)
            qr = np.zeros(num, np.int16); qo = np.zeros(num, np.int16)
            nr = get("quant", C.c_uint32, [P, P, P, P, I, I, I])(ptr(coef), ptr(qc), ptr(dur), ptr(qr), qbits, add, num)
            no = O.orc_quant(ptr(coef), ptr(qc), ptr(duo), ptr(qo), qbits, add, num)
            assert nr == no and same(ref_out(qr), qo) and same(ref_out(dur), duo)
            nr = get("nquant", C.c_uint32, [P, P, P, I, I, I])(ptr(coef), ptr(qc), ptr(qr), qbits, add, num)
            no = O.orc_nquant(ptr(coef), ptr(qc), ptr(qo), qbits, add, num)
            assert nr == no and same(ref_out(qr), qo)
            scale = int(rng.integers(1, 32768)); shift = int(rng.integers(1, 11))
            get("dequant_normal", None, [P, P, I, I, I])(ptr(coef), ptr(qr), num, scale, shift)
            O.orc_dequant_normal(ptr(coef), ptr(qo), num, scale, shift)
            assert same(ref_out(qr), qo)
            dq = rng.integers(1, 1 << 12, num).astype(np.int32)
            for per in (0, 3, 9):
                sh = int(rng.integers(1, 7))
                get("dequant_scaling", None, [P, P, P, I, I, I])(ptr(coef), ptr(dq), ptr(qr), num, per, sh)
                O.orc_dequant_scaling(ptr(coef), ptr(dq), ptr(qo), num, per, sh)
                assert same(ref_out(qr), qo)
            c1 = coef.copy(); c2 = coef.copy()
            rs1 = np.zeros(num, np.uint32); rs2 = np.zeros(num, np.uint32)
            off = rng.integers(0, 300, num).astype(np.uint16)
            get("denoiseDct", None, [P, P, P, I])(ptr(c1), ptr(rs1), ptr(off), num)
            O.orc_denoise_dct(ptr(c2), ptr(rs2), ptr(off), num)
            assert same(ref_out(c1), c2) and same(ref_out(rs1), rs2)
    # cuTree propagateCost (pixel.cpp:914-940): double arithmetic, incl. the degenerate intraCost == 0 entries (0/0 -> INT_MIN)
    for it in range(3):
        n = int(rng.integers(16, 400))
        pin = rng.integers(0, 65536, n).astype(np.uint16); intra = rng.integers(0 if it else 1, 1 << 15, n).astype(np.int32)
        inter = rng.integers(0, 65536, n).astype(np.uint16); invq = rng.integers(1, 1024, n).astype(np.int32)
        if kind == "max":
            intra[:] = (1 << 15) - 1; pin[:] = 65535
        fps = np.array([256.0 * (0.01 + 0.33 * it)], np.float64)
        d1 = np.full(n, -3, np.int32); d2 = np.full(n, -3, np.int32)
        get("propagateCost", None, [P, P, P, P, P, P, I])(ptr(d1), ptr(pin), ptr(intra), ptr(inter), ptr(invq), ptr(fps), n)
        O.orc_propagate_cost(ptr(d2), ptr(pin), ptr(intra), ptr(inter), ptr(invq), ptr(fps), n)
        assert same(ref_out(d1), d2), (it, np.nonzero(d1 != d2)[0][:5])


def check_integral(get, O, depth, ref_out=lambda v: v):
    """SEA integral-plane primitives (framefilter.cpp:39-143): integral_inith[k] / integral_initv[k], k = IntegralSize
    (4, 8, 12, 16, 24, 32); uint32 wrap-around sums, rows as FrameFilter::computeMEIntegral hands them over."""
    rng = np.random.default_rng(33 + depth)
    dt = pixel_dtype(depth)
    for k, n in enumerate((4, 8, 12, 16, 24, 32)):
        for stride in (56, 64, 200):
            pix = rng.integers(0, 1 << depth, stride + 64).astype(dt)
            base = rng.integers(0, 1 << 32, stride * (n + 3), dtype=np.uint64).astype(np.uint32)
            a, b = base.copy(), base.copy()
            get("integral_inith", None, [P, P, IP], k)(ptr(a, stride), ptr(pix), IP(stride))
            O.orc_integral_inith(ptr(b, stride), ptr(pix), IP(stride), n)
            assert same(ref_out(a), b), ("inith", n, stride)
            a, b = base.copy(), base.copy()
            get("integral_initv", None, [P, IP], k)(ptr(a, stride), IP(stride))
            O.orc_integral_initv(ptr(b, stride), IP(stride), n)
            assert same(ref_out(a), b), ("initv", n, stride)


def check_intra(get, O, depth, kind, ref_out=lambda v: v):
    rng = np.random.default_rng(6)
    dt = pixel_dtype(depth)
    for cu, n in enumerate(LUMA_CU[:4]):
        for it in range(4):
            nb = fixtures(rng, depth, (4 * n + 1 + 16,), kind)
            fr = np.zeros(4 * n + 1 + 16, dt); fo = np.zeros(4 * n + 1 + 16, dt)
            get("cu.intra_filter", None, [P, P], cu)(ptr(nb), ptr(fr))
            O.orc_intra_filter(ptr(nb), ptr(fo), n)
            assert same(ref_out(fr), fo)
            for mode in range(35):
                for bf in (0, 1):
                    dr = np.zeros((n, 64), dt); do = np.zeros((n, 64), dt)
                    get("cu.intra_pred", None, [P, IP, P, I, I], cu, mode)(ptr(dr), 64, ptr(nb), mode, bf)
                    O.orc_intra_pred(ptr(do), IP(64), ptr(nb), mode, bf, n)
                    assert same(ref_out(dr), do), (n, mode, bf)
            for bl in (0, 1):
                ar = np.zeros(33 * n * n, dt); ao = np.zeros(33 * n * n, dt)
                get("cu.intra_pred_allangs", None, [P, P, P, I], cu)(ptr(ar), ptr(nb), ptr(fr), bl)
                O.orc_intra_pred_allangs(ptr(ao), ptr(nb), ptr(fo), bl, n)
                assert same(ref_out(ar), ao), (n, bl)
