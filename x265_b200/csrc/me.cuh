// x265_b200/csrc/me.cuh -- motion-estimation class: one warp replays one
// MotionEstimate::motionEstimate() call (/root/reference/source/encoder/motion.cpp:739-1569)
// bit-exactly: MVP / zero / candidate pre-checks (:771-814), DIA (:822-846), HEX (:848-945),
// STAR (:362-604, :1132-1240 incl. the raster refinement and its `tmv << 3` quirk), sub-pel
// refinement by workload[subme] (:48-58, :1449-1558) through subpelCompare (:1571-1598, luma) or
// the lowres qpel path (common/lowres.h:94-120).
//
// Parallelism: (PUs x refs x CTUs) jobs per launch, one warp per job, and INSIDE a job every burst
// of independent candidates (the 4/8/16 points of a star level, 32 raster points, the 4/8 sub-pel
// directions of a refinement round) is evaluated by the 32 lanes at once -- (candidate, pixel-word)
// pairs are spread over the lanes -- and then folded in the reference's sequential order, so the
// decisions are identical.  Costs are warp-uniform after each fold: all lanes take the same branches.
#pragma once
#include "common.cuh"
#include "pixelcmp.cuh"
#include "interp.cuh"

#define ME_BAND 16                         // rows of prediction staged per pass
#define ME_MID_ROWS (ME_BAND + 7)

struct MeShared                            // per-warp scratch
{
    int16_t mid[ME_MID_ROWS * 64];         // hps(rowExt) intermediate of one band (or 4 small candidates)
    uint16_t pred[ME_BAND * 64];           // predicted band (or 4 small candidates)
};

template <typename P>
struct MeCtx
{
    const P* fenc;  int fstride;           // fenc block origin (plane + offset)
    const P* ref[4]; int rstride;          // ref plane(s) + offset
    const uint16_t* mvc;                   // centred mvcost table
    int mvpx, mvpy;
    int minx, miny, maxx, maxy;            // full-pel bounds
    int w, h, lgw, lane, lowres;
    bool pow2;                             // w and h are powers of two (all 2Nx2N / rect PUs); AMP sizes take the generic paths
    int nw, lgnw, lgwpr;                   // words per PU, log2, log2(words per row)
    int lgsegw;                            // log2 words per lane segment (16 B when the fenc rows allow vector loads)
    int ppitch;                            // byte distance between quarter-pel phase planes (0: none, candidates interpolate)
    MeShared* sm;
};

// Quarter-pel phase planes (analyser.cuh, k_luma_phase_planes): the reference allocation holds 16 planes ppitch bytes
// apart; plane (yFrac << 2) | xFrac is the reference predicted at that phase (luma_hpp / luma_vpp / luma_hvpp), so a
// sub-pel candidate (qx, qy) is a full-pel block of plane ((qy & 3) << 2) | (qx & 3) at (qx >> 2, qy >> 2).
template <typename P>
__device__ __forceinline__ int me_qpel_off(const MeCtx<P>& c, int qx, int qy)       // byte offset from c.ref[0]
{
    return ((((qy & 3) << 2) | (qx & 3)) * c.ppitch) + ((qy >> 2) * c.rstride + (qx >> 2)) * (int)sizeof(P);
}
template <typename P>
__device__ __forceinline__ const P* me_qpel_ptr(const MeCtx<P>& c, int qx, int qy)
{
    return (const P*)((const uint8_t*)c.ref[0] + me_qpel_off(c, qx, qy));
}

template <typename P>
__device__ __forceinline__ int me_mvcost(const MeCtx<P>& c, int qx, int qy)
{
    return (uint16_t)(__ldg(c.mvc + (qx - c.mvpx)) + __ldg(c.mvc + (qy - c.mvpy)));
}

template <typename P>
__device__ __forceinline__ void me_yx(const MeCtx<P>& c, int i, int& y, int& x)
{
    if (c.pow2) { y = i >> c.lgw; x = i & (c.w - 1); }
    else        { y = i / c.w; x = i - y * c.w; }
}

__device__ __forceinline__ uint32_t ld_unaligned32(uintptr_t a)
{
    const uint32_t* ap = (const uint32_t*)(a & ~(uintptr_t)3);
    const uint32_t sh = (uint32_t)(a & 3) * 8;
    uint32_t lo = __ldg(ap);
    return sh ? __funnelshift_r(lo, __ldg(ap + 1), sh) : lo;
}

template <typename P> __device__ __forceinline__ int sad_word(uint32_t a, uint32_t b, int acc)
{
    return sizeof(P) == 1 ? (int)(__vsadu4(a, b) + (uint32_t)acc) : (int)(__vsadu2(a, b) + (uint32_t)acc);
}
// SAD of N (<= 16) words.  8-bit: N VABSDIFF4 with accumulate.  16-bit: sm_100a has no packed absolute-difference-and-add
// for halves (__vsadu2 is ~8 instructions); max - min per half IS native (VIMNMX.U16x2) and cannot borrow, so the N packed
// differences are summed in the two 16-bit lanes (<= 16 * 1023 each for 10-bit pixels, <= 16 * 4095 for 12-bit) and folded
// once: about 3 instructions per word instead of 8.
template <typename P, int N>
__device__ __forceinline__ int sad_words(const uint32_t (&a)[N], const uint32_t (&b)[N], int acc)
{
    if (sizeof(P) == 1)
    {
#pragma unroll
        for (int k = 0; k < N; k++) acc = (int)(__vsadu4(a[k], b[k]) + (uint32_t)acc);
        return acc;
    }
    uint32_t t = 0;
#pragma unroll
    for (int k = 0; k < N; k++) t += __vmaxu2(a[k], b[k]) - __vminu2(a[k], b[k]);
    return acc + (int)(t & 0xffffu) + (int)(t >> 16);
}

// ---- full-pel SAD of up to 32 candidate positions at once (pow2 PUs) -----------------------------
// The PU is cut into row segments of SEGW words (16 bytes when the rows are wide and aligned enough).
// With n candidates in the burst, lpc = 32 / pow2ceil(n) lanes share one candidate (capped by the number
// of segments); the lpc lanes split the PU's columns first and its rows second, so a lane walks a fixed
// set of columns down the rows with incremental addresses.  Per segment: one vector load of fenc (the
// same address in every candidate group: one L1 broadcast), SEGW+1 aligned words of the reference
// funnel-shifted to the candidate's byte phase, SEGW VABSDIFF4.ACC.  All candidates of a burst are in
// flight together; one xor-shuffle tree per burst folds the lanes of each candidate.
// `offB` = byte offset of lane i's candidate from `base` (lanes >= n ignored).  Result in lane i < n.
template <typename P, int LGSEGW>
__device__ __forceinline__ int me_sad_multi_t(const MeCtx<P>& c, const uint8_t* __restrict__ base, int n, int offB)
{
    constexpr int SEGW = 1 << LGSEGW;
    const int lane = c.lane;
    const int lgn = n <= 1 ? 0 : 32 - __clz(n - 1);
    const int lgnseg = c.lgnw - LGSEGW, lgspr = c.lgwpr - LGSEGW;          // log2 segments per PU / per row
    const int lglpc = min(5 - lgn, lgnseg);
    const int lgcols = min(lglpc, lgspr), lgrows = lglpc - lgcols;         // lanes of a candidate: 2^lgcols across, 2^lgrows down
    const int sub = lane & ((1 << lglpc) - 1);
    const int ob = __shfl_sync(0xffffffffu, offB, min(lane >> lglpc, n - 1));
    const uintptr_t cptr = (uintptr_t)base + (intptr_t)ob;                 // my candidate's block origin; any byte phase
    const unsigned sh = ((unsigned)cptr & 3u) * 8u;
    const int rsB = c.rstride * (int)sizeof(P), fsB = c.fstride * (int)sizeof(P);
    const int subcol = sub & ((1 << lgcols) - 1), subrow = sub >> lgcols;
    // 16- and 8-byte segments read the reference as 8-byte aligned LDG.64 (three / two instead of five / three LDG.32: the
    // kernel sits at the LSU issue floor) and pick the word phase with one select per word; row pitch and column step are
    // multiples of 8 bytes, so the phase is the same for every segment of the walk
    const bool hi8 = SEGW >= 2 && ((unsigned)cptr & 4u) != 0;
    const uint8_t* rrow = (const uint8_t*)(cptr & ~(uintptr_t)(SEGW >= 2 ? 7 : 3)) + subrow * rsB + subcol * (SEGW * 4);
    const uint8_t* frow = (const uint8_t*)c.fenc + subrow * fsB + subcol * (SEGW * 4);
    const int rowStepR = rsB << lgrows, rowStepF = fsB << lgrows, colStep = (SEGW * 4) << lgcols;
    const int nrows = c.h >> lgrows, ncols = 1 << (lgspr - lgcols);
    int acc = 0;
    // columns outside (1..8 iterations), rows inside: the long dimension is the unrolled one
    for (int jc = 0; jc < ncols; jc++, rrow += colStep, frow += colStep)
    {
        const uint8_t* rp = rrow; const uint8_t* fp = frow;
#pragma unroll 2
        for (int i = 0; i < nrows; i++, rp += rowStepR, fp += rowStepF)
        {
            const uint32_t* ap = (const uint32_t*)rp;
            if (SEGW == 4)
            {
                const uint4 f = __ldg((const uint4*)fp);
                const uint2 a0 = __ldg((const uint2*)rp), a1 = __ldg((const uint2*)rp + 1), a2 = __ldg((const uint2*)rp + 2);
                const uint32_t w0 = hi8 ? a0.y : a0.x, w1 = hi8 ? a1.x : a0.y, w2 = hi8 ? a1.y : a1.x, w3 = hi8 ? a2.x : a1.y, w4 = hi8 ? a2.y : a2.x;
                const uint32_t fa[4] = { f.x, f.y, f.z, f.w };
                const uint32_t ra[4] = { __funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh), __funnelshift_r(w2, w3, sh), __funnelshift_r(w3, w4, sh) };
                acc = sad_words<P, 4>(fa, ra, acc);
            }
            else if (SEGW == 2)
            {
                const uint2 f = __ldg((const uint2*)fp);
                const uint2 a0 = __ldg((const uint2*)rp), a1 = __ldg((const uint2*)rp + 1);
                const uint32_t w0 = hi8 ? a0.y : a0.x, w1 = hi8 ? a1.x : a0.y, w2 = hi8 ? a1.y : a1.x;
                const uint32_t fa[2] = { f.x, f.y };
                const uint32_t ra[2] = { __funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh) };
                acc = sad_words<P, 2>(fa, ra, acc);
            }
            else
            {
                const uint32_t f = __ldg((const uint32_t*)fp);
                acc = sad_word<P>(f, __funnelshift_r(__ldg(ap), __ldg(ap + 1), sh), acc);
            }
        }
    }
    for (int o = 1; o < (1 << lglpc); o <<= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    return __shfl_sync(0xffffffffu, acc, (lane << lglpc) & 31);
}

template <typename P>
__device__ __forceinline__ int me_sad_multi(const MeCtx<P>& c, const uint8_t* __restrict__ base, int n, int offB)
{
#ifdef ME_SEG_PER_BURST
    // experiment (DESIGN.md section 8 item 1, build with -DME_SEG_PER_BURST): narrow the lane segment so that the lanes sharing a
    // candidate fill one row before they spread over rows (fewer distinct lines per request for small-PU star bursts)
    const int lgn = n <= 1 ? 0 : 32 - __clz(n - 1);
    const int lgseg = min(c.lgsegw, max(0, c.lgwpr - (5 - lgn)));
    if (lgseg == 2) return me_sad_multi_t<P, 2>(c, base, n, offB);
    if (lgseg == 1) return me_sad_multi_t<P, 1>(c, base, n, offB);
    return me_sad_multi_t<P, 0>(c, base, n, offB);
#else
    if (c.lgsegw == 2) return me_sad_multi_t<P, 2>(c, base, n, offB);
    if (c.lgsegw == 1) return me_sad_multi_t<P, 1>(c, base, n, offB);
    return me_sad_multi_t<P, 0>(c, base, n, offB);
#endif
}

// SAD of the fenc block against ONE reference position (element pointer, rows may be unaligned); all lanes get it.
template <typename P>
__device__ __noinline__ int me_sad_direct(const MeCtx<P>& c, const P* __restrict__ r)
{
    if (c.pow2) return __shfl_sync(0xffffffffu, me_sad_multi(c, (const uint8_t*)r, 1, 0), 0);
    // AMP sizes (12/24/48): generic word walk
    const uintptr_t rbase = (uintptr_t)r;
    int acc = 0;
    const int wprg = (c.w * (int)sizeof(P)) >> 2, nwg = wprg * c.h;
    for (int wd = c.lane; wd < nwg; wd += 32)
    {
        int row = wd / wprg, col = wd - row * wprg;
        uint32_t f = __ldg((const uint32_t*)((const uint8_t*)c.fenc + ((size_t)row * c.fstride) * sizeof(P) + col * 4));
        acc = sad_word<P>(f, ld_unaligned32(rbase + ((size_t)row * c.rstride) * sizeof(P) + col * 4), acc);
    }
    return warp_sum(acc);
}

// SAD of up to 32 blocks at once: lane i (< n) owns the block at byte offset offB from c.ref[0]; result in lane i
template <typename P>
__device__ __forceinline__ int me_sad_points(const MeCtx<P>& c, int n, int offB)
{
    const uint8_t* rbase = (const uint8_t*)c.ref[0];
    int mysad = 0;
    if (c.pow2) mysad = me_sad_multi(c, rbase, n, offB);
    else
    {
        for (int p = 0; p < n; p++)
        {
            const int offp = __shfl_sync(0xffffffffu, offB, p);
            const int v = me_sad_direct(c, (const P*)(rbase + offp));
            if (c.lane == p) mysad = v;
        }
    }
    return mysad;
}

// Full-pel SAD + mvcost of up to 32 candidate positions at once.  Lane i (< n) owns candidate i:
// (px, py) in full-pel units relative to the block; returns that candidate's cost in lane i.
// x8: the raster quirk (motion.cpp:1194: mvcost(tmv << 3) for every 4th column).
template <typename P>
__device__ __forceinline__ int me_eval_points(const MeCtx<P>& c, int n, int px, int py, bool x8)
{
    const int mysad = me_sad_points(c, n, (py * c.rstride + px) * (int)sizeof(P));
    int cost = 0x7fffffff;
    if (c.lane < n) cost = mysad + (x8 ? me_mvcost(c, px * 8, py * 8) : me_mvcost(c, px * 4, py * 4));
    return cost;
}


// tile distortions kept out of line: the job loop is instruction-cache bound, one copy of the unrolled
// Hadamard instead of six is worth more than the call overhead (measured: profiles/me_r1 notes)
template <typename PA, typename PB>
__device__ __forceinline__ int me_tile8x4(const PA* pf, int sf, const PB* pp, int sp)
{
    return (had4x4_abs(pf, sf, pp, sp) + had4x4_abs(pf + 4, sf, pp + 4, sp)) >> 1;
}
template <typename PA, typename PB>
__device__ __forceinline__ int me_tile4x4(const PA* pf, int sf, const PB* pp, int sp)
{
    return had4x4_abs(pf, sf, pp, sp) >> 1;
}

// keep only the valid candidates, preserving order: returns n and moves candidate k to lane k.
// `cnt` = number of generated candidates (lanes >= cnt are invalid by construction).
__device__ __forceinline__ int me_compact(bool valid, int cnt, int& a, int& b, int& c2, int& d)
{
    const unsigned m = __ballot_sync(0xffffffffu, valid);
    if (m == ((cnt >= 32) ? 0xffffffffu : ((1u << cnt) - 1u))) return cnt;      // common case: nothing to drop
    const int lane = threadIdx.x & 31;
    // lane k takes the candidate of the k-th set bit: strip the k lowest set bits, then find-first-set
    unsigned t = m;
    for (int k = 0; k < lane && t; k++) t &= t - 1;
    const int src = t ? (__ffs(t) - 1) : 0;
    a = __shfl_sync(0xffffffffu, a, src); b = __shfl_sync(0xffffffffu, b, src);
    c2 = __shfl_sync(0xffffffffu, c2, src); d = __shfl_sync(0xffffffffu, d, src);
    return __popc(m);
}

// cost of a band of prediction held in c.sm->pred (stride 64) against fenc rows [y0, y0+rows)
template <typename P>
__device__ __forceinline__ int me_band_cost(const MeCtx<P>& c, int y0, int rows, bool satd)
{
    const uint16_t* pr = c.sm->pred;
    const P* f = c.fenc + (size_t)y0 * c.fstride;
    int acc = 0;
    if (!satd)
    {
        const int n = rows * c.w;
        for (int i = c.lane; i < n; i += 32)
        {
            int y, x; me_yx(c, i, y, x);
            acc += abs((int)f[y * c.fstride + x] - (int)pr[y * 64 + x]);
        }
    }
    else if (!c.pow2)
    {   // AMP sizes: 8x4 tiles when w % 8 == 0, else 4x4 tiles (pixel.cpp:1134-1158)
        const int tw = (c.w & 7) == 0 ? 8 : 4, tpr = c.w / tw, nt = tpr * (rows >> 2);
        for (int t = c.lane; t < nt; t += 32)
        {
            int ty = t / tpr, tx = t - ty * tpr;
            const P* pf = f + (ty * 4) * c.fstride + tx * tw; const uint16_t* pp = pr + (ty * 4) * 64 + tx * tw;
            if (tw == 8) acc += me_tile8x4(pf, c.fstride, pp, 64);
            else         acc += had4x4_abs(pf, c.fstride, pp, 64) >> 1;
        }
    }
    else if (c.w >= 8)
    {
        const int lgtw = c.lgw - 3, nt = (rows >> 2) << lgtw;
        for (int t = c.lane; t < nt; t += 32)
        {
            int ty = t >> lgtw, tx = t & ((1 << lgtw) - 1);
            const P* pf = f + (ty * 4) * c.fstride + tx * 8; const uint16_t* pp = pr + (ty * 4) * 64 + tx * 8;
            acc += me_tile8x4(pf, c.fstride, pp, 64);
        }
    }
    else
    {
        const int nt = rows >> 2;                    // w == 4: one 4x4 tile per 4 rows
        for (int t = c.lane; t < nt; t += 32)
            acc += me_tile4x4(f + (t * 4) * c.fstride, c.fstride, pr + (t * 4) * 64, 64);
    }
    return acc;           // un-reduced partial (caller reduces once)
}

// subpelCompare (motion.cpp:1571-1598) for ONE candidate: luma_hpp / luma_vpp / luma_hvpp, then cmp.
template <typename P>
__device__ __forceinline__ int me_subpel_compare_t(const MeCtx<P>& c, int qx, int qy, bool satd)
{
    constexpr int DEPTH = PixTraits<P>::depth;
    const P* r = c.ref[0] + (qx >> 2) + (ptrdiff_t)(qy >> 2) * c.rstride;
    const int xf = qx & 3, yf = qy & 3;
    if (!(xf | yf))
    {
        if (!satd) return me_sad_direct(c, r);
        return warp_satd(c.fenc, c.fstride, r, c.rstride, c.w, c.h, c.lane);
    }
    const int16_t* cx = c_lumaFilter[xf];
    const int16_t* cy = c_lumaFilter[yf];
    int acc = 0;
    for (int y0 = 0; y0 < c.h; y0 += ME_BAND)
    {
        const int rows = min(ME_BAND, c.h - y0);
        __syncwarp();
        if (!yf)
        {
            for (int i = c.lane; i < rows * c.w; i += 32)
            {
                int y, x; me_yx(c, i, y, x);
                const P* s = r + (ptrdiff_t)(y0 + y) * c.rstride + x - 3;
                c.sm->pred[y * 64 + x] = (uint16_t)interp_finish<DEPTH>(me_hsum8(s, cx, xf), 0);
            }
        }
        else if (!xf)
        {
            for (int i = c.lane; i < rows * c.w; i += 32)
            {
                int y, x; me_yx(c, i, y, x);
                const P* s = r + (ptrdiff_t)(y0 + y - 3) * c.rstride + x;
                int sum = 0;
#pragma unroll
                for (int k = 0; k < 8; k++) sum += (int)s[(ptrdiff_t)k * c.rstride] * cy[k];
                c.sm->pred[y * 64 + x] = (uint16_t)interp_finish<DEPTH>(sum, 0);
            }
        }
        else
        {
            const int mrows = rows + 7;
            for (int i = c.lane; i < mrows * c.w; i += 32)
            {
                int y, x; me_yx(c, i, y, x);
                const P* s = r + (ptrdiff_t)(y0 + y - 3) * c.rstride + x - 3;
                c.sm->mid[y * 64 + x] = (int16_t)interp_finish<DEPTH>(me_hsum8(s, cx, xf), 1);
            }
            __syncwarp();
            for (int i = c.lane; i < rows * c.w; i += 32)
            {
                int y, x; me_yx(c, i, y, x);
                int sum = 0;
#pragma unroll
                for (int k = 0; k < 8; k++) sum += (int)c.sm->mid[(y + k) * 64 + x] * cy[k];
                c.sm->pred[y * 64 + x] = (uint16_t)interp_finish<DEPTH>(sum, 2);
            }
        }
        __syncwarp();
        acc += me_band_cost(c, y0, rows, satd);
    }
    return warp_sum(acc);
}

// ---- sub-pel evaluation of SMALL PUs (pow2, w and h <= 16): one lane = one 8-pixel (4 for w = 4) row segment ----
// (row helpers me_hrow / me_vcol / me_vmid: interp.cuh)
// NPX pixels of a source row segment as ints: one aligned vector load when the rows allow it
template <typename P, int NPX>
__device__ __forceinline__ void me_load_fenc(const MeCtx<P>& c, const P* __restrict__ f, int (&v)[NPX])
{
    constexpr int NWD = NPX * (int)sizeof(P) / 4;
    if ((4 << c.lgsegw) >= NPX * (int)sizeof(P))
    {
        uint32_t w[NWD];
        if (NWD == 1) w[0] = __ldg((const uint32_t*)f);
        else if (NWD == 2) { const uint2 t = __ldg((const uint2*)f); w[0] = t.x; w[NWD - 1] = t.y; }
        else { const uint4 t = __ldg((const uint4*)f); w[0] = t.x; w[1 % NWD] = t.y; w[2 % NWD] = t.z; w[3 % NWD] = t.w; }
#pragma unroll
        for (int x = 0; x < NPX; x++)
            v[x] = sizeof(P) == 1 ? (int)((w[x >> 2] >> (8 * (x & 3))) & 255u) : (int)((w[x >> 1] >> (16 * (x & 1))) & 65535u);
    }
    else
    {
#pragma unroll
        for (int x = 0; x < NPX; x++) v[x] = (int)__ldg(f + x);
    }
}

// N consecutive pixels at any alignment as ints (forward declaration: defined with the chroma helpers below)
template <typename P, int N>
__device__ __forceinline__ void me_ld_px(const P* __restrict__ p, int (&v)[N]);

// Up to 4 sub-pel candidates of a SMALL PU, lane i (< n <= 4) owns candidate i (qx, qy) and gets its distortion.
// Per candidate the arithmetic is exactly subpelCompare's (motion.cpp:1571-1598: luma_hpp / luma_vpp / luma_hvpp
// = hps(rowExt) + vsp, ipfilter.cpp:79-369) followed by sad or satd (8x4 tiles, 4x4 for w = 4; pixel.cpp:263-297).
// Mapping: lane = (candidate slot, segment, row): a PU of h rows and w/8 segments takes h * w/8 lanes, so 4
// candidates of an 8x8 run at once (2 of a 16x8, 1 of a 16x16).  hv candidates first write their h+7 horizontally
// filtered rows to shared memory (one row segment per lane-task), then every lane produces ITS row of the
// prediction in registers, differences it against the source row, does the horizontal half of the 4x4 Hadamards
// in registers and the vertical half with two xor-shuffle butterflies over the 4 lanes of a tile.
// PL: the candidates are read from the quarter-pel phase planes (no filtering, no shared memory).
template <typename P, int NPX, bool PL>
__device__ __forceinline__ int me_subpel_small_t(const MeCtx<P>& c, int n, int qx, int qy, bool satd)
{
    constexpr int DEPTH = PixTraits<P>::depth;
    const int lane = c.lane;
    const int lgsegs = NPX == 8 ? c.lgw - 3 : 0;                 // log2 segments per row
    const int lgh = 31 - __clz(c.h);
    const int lglpc = lgh + lgsegs, lpc = 1 << lglpc;            // lanes per candidate: 4 .. 32
    const int cpp = min(4, 32 >> lglpc);                         // candidate slots per pass
    const int midPer = (c.h + 7) * c.w;                          // int16 elements of one candidate's intermediate
    const int tasksPer = (c.h + 7) << lgsegs;
    int16_t* mid = c.sm->mid;
    int out = 0;
    for (int base = 0; base < n; base += cpp)
    {
        const int live_n = min(cpp, n - base);
        __syncwarp();
        // ---- stage 1: horizontally filtered rows of the hv candidates ----
        for (int t0 = 0; !PL && t0 < live_n * tasksPer; t0 += 32)
        {
            const int t = t0 + lane;
            const int tci = min((int)(t >= tasksPer) + (int)(t >= 2 * tasksPer) + (int)(t >= 3 * tasksPer), live_n - 1);
            const int tt = t - tci * tasksPer;
            const int tqx = __shfl_sync(0xffffffffu, qx, base + tci), tqy = __shfl_sync(0xffffffffu, qy, base + tci);
            const int txf = tqx & 3, tyf = tqy & 3;
            if (t < live_n * tasksPer && txf && tyf)
            {
                const int mrow = tt >> lgsegs, seg = tt & ((1 << lgsegs) - 1);
                const P* s = c.ref[0] + (tqx >> 2) + (ptrdiff_t)((tqy >> 2) - 3 + mrow) * c.rstride + seg * 8;
                int sum[NPX];
                me_hrow<P, NPX>(s, txf, sum);
                uint32_t pk[NPX / 2];
#pragma unroll
                for (int i = 0; i < NPX / 2; i++)
                    pk[i] = ((uint32_t)interp_finish<DEPTH>(sum[2 * i], 1) & 0xffffu) | ((uint32_t)interp_finish<DEPTH>(sum[2 * i + 1], 1) << 16);
                int16_t* d = mid + tci * midPer + mrow * c.w + seg * 8;
                if (NPX == 8) *(uint4*)d = make_uint4(pk[0], pk[1], pk[NPX / 2 - 2], pk[NPX / 2 - 1]);
                else          *(uint2*)d = make_uint2(pk[0], pk[NPX / 2 - 1]);
            }
        }
        __syncwarp();
        // ---- stage 2: my row segment of my candidate's prediction ----
        const int ci = lane >> lglpc, sub = lane & (lpc - 1);
        const bool live = ci < live_n;
        const int cand = base + min(ci, live_n - 1);
        const int mqx = __shfl_sync(0xffffffffu, qx, cand), mqy = __shfl_sync(0xffffffffu, qy, cand);
        const int xf = mqx & 3, yf = mqy & 3;
        const int row = sub & (c.h - 1), seg = sub >> lgh;
        int d[NPX];
        if (live)
        {
            const P* r = c.ref[0] + (mqx >> 2) + (ptrdiff_t)((mqy >> 2) + row) * c.rstride + seg * 8;
            int pr[NPX];
            if (PL) me_ld_px<P, NPX>(me_qpel_ptr(c, mqx, mqy) + (ptrdiff_t)row * c.rstride + seg * 8, pr);
            else if (!(xf | yf))
            {
#pragma unroll
                for (int x = 0; x < NPX; x++) pr[x] = (int)__ldg(r + x);
            }
            else if (!yf)
            {
                me_hrow<P, NPX>(r, xf, pr);
#pragma unroll
                for (int x = 0; x < NPX; x++) pr[x] = interp_finish<DEPTH>(pr[x], 0);
            }
            else if (!xf)
            {
                me_vcol<P, NPX>(r - 3 * (ptrdiff_t)c.rstride, c.rstride, yf, pr);
#pragma unroll
                for (int x = 0; x < NPX; x++) pr[x] = interp_finish<DEPTH>(pr[x], 0);
            }
            else
            {
                me_vmid<NPX>(mid + min(ci, live_n - 1) * midPer + row * c.w + seg * 8, c.w, yf, pr);
#pragma unroll
                for (int x = 0; x < NPX; x++) pr[x] = interp_finish<DEPTH>(pr[x], 2);
            }
            int fv[NPX];
            me_load_fenc<P, NPX>(c, c.fenc + (ptrdiff_t)row * c.fstride + seg * 8, fv);
#pragma unroll
            for (int x = 0; x < NPX; x++) d[x] = fv[x] - pr[x];
        }
        else
        {
#pragma unroll
            for (int x = 0; x < NPX; x++) d[x] = 0;
        }
        // ---- stage 3: distortion ----
        int part = 0;
        if (!satd)
        {
#pragma unroll
            for (int x = 0; x < NPX; x++) part += abs(d[x]);
            for (int o = 1; o < lpc; o <<= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
        }
        else
        {
#pragma unroll
            for (int x = 0; x < NPX; x += 4) had4(d[x], d[x + 1], d[x + 2], d[x + 3]);
#pragma unroll
            for (int st = 1; st <= 2; st <<= 1)
            {
                const bool up = (lane & st) != 0;
#pragma unroll
                for (int x = 0; x < NPX; x++)
                {
                    const int o = __shfl_xor_sync(0xffffffffu, d[x], st);
                    d[x] = up ? o - d[x] : o + d[x];
                }
            }
#pragma unroll
            for (int x = 0; x < NPX; x++) part += abs(d[x]);
            part += __shfl_xor_sync(0xffffffffu, part, 1);
            part += __shfl_xor_sync(0xffffffffu, part, 2);
            part = (lane & 3) ? 0 : (part >> 1);                    // one 8x4 (4x4) tile per 4 lanes, halved per tile
            for (int o = 4; o < lpc; o <<= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
        }
        const int v = __shfl_sync(0xffffffffu, part, ((lane - base) << lglpc) & 31);
        if (lane >= base && lane < base + live_n) out = v;
    }
    return out;
}

// One sub-pel candidate of a LARGE pow2 PU (w >= 8, more than 32 row segments), same lane = row-segment scheme in
// bands of 16 rows: the band's 23 horizontally filtered rows go through shared memory (hv only), every lane then
// produces row segments of the prediction in registers, 32 at a time.  All lanes get the distortion.
// 8 reference pixels of a row at any byte phase as ints (forward declaration: defined with the lowres helpers below)
template <typename P>
__device__ __forceinline__ void me_load_row8(const P* __restrict__ p, int (&v)[8]);

// LARGE pow2 PUs (w > 16 or h > 16; w >= 8): a lane owns an 8x4 UNIT = 4 consecutive rows of an 8-pixel strip, i.e.
// exactly one 8x4 SATD tile: the Hadamard is entirely in the lane's registers (no shuffles) and the vertical filters
// re-use their source rows (11 rows feed 4 output rows: me_vcol4 / me_vmid4).  The PU is processed in bands of
// BR = min(h, 1024 / w) rows (a full warp of units for w = 64 / 32 / 16 with h >= 16 / 32 / 64); hv candidates first
// write the band's BR + 7 horizontally filtered rows to shared memory (one row segment per lane-task).
// PL: the candidate is a full-pel block of its quarter-pel phase plane (every candidate takes the unit path of xf = yf = 0).
template <typename P, bool PL>
__device__ __forceinline__ int me_subpel_big(const MeCtx<P>& c, int qx, int qy, bool satd)
{
    constexpr int DEPTH = PixTraits<P>::depth;
    const int lane = c.lane;
    const int lgsegs = c.lgw - 3, segs = 1 << lgsegs;
    const int xf = PL ? 0 : qx & 3, yf = PL ? 0 : qy & 3;
    const P* r0 = PL ? me_qpel_ptr(c, qx, qy) : c.ref[0] + (qx >> 2) + (ptrdiff_t)(qy >> 2) * c.rstride;
    if (!(xf | yf) && !satd) return me_sad_direct(c, r0);             // full-pel SAD: the word-wise SAD core
    int16_t* mid = c.sm->mid;
    const int BR = min(c.h, 1024 >> c.lgw);
    const int units = (BR >> 2) << lgsegs;
    int acc = 0;
    for (int y0 = 0; y0 < c.h; y0 += BR)
    {
        if (xf && yf)
        {
            __syncwarp();
            const int tasks = (BR + 7) << lgsegs;
            for (int t = lane; t < tasks; t += 32)
            {
                const int mrow = t >> lgsegs, seg = t & (segs - 1);
                int sum[8];
                me_hrow<P, 8>(r0 + (ptrdiff_t)(y0 - 3 + mrow) * c.rstride + seg * 8, xf, sum);
                uint32_t pk[4];
#pragma unroll
                for (int i = 0; i < 4; i++)
                    pk[i] = ((uint32_t)interp_finish<DEPTH>(sum[2 * i], 1) & 0xffffu) | ((uint32_t)interp_finish<DEPTH>(sum[2 * i + 1], 1) << 16);
                *(uint4*)(mid + mrow * c.w + seg * 8) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
            }
            __syncwarp();
        }
        for (int u = lane; u < units; u += 32)
        {
            const int seg = u & (segs - 1), row = (u >> lgsegs) << 2;          // first row of the unit inside the band
            const P* r = r0 + (ptrdiff_t)(y0 + row) * c.rstride + seg * 8;
            int d[4][8];
            if (!(xf | yf))
            {
#pragma unroll
                for (int y = 0; y < 4; y++) me_load_row8<P>(r + (ptrdiff_t)y * c.rstride, d[y]);
            }
            else if (!yf)
            {
#pragma unroll
                for (int y = 0; y < 4; y++)
                {
                    me_hrow<P, 8>(r + (ptrdiff_t)y * c.rstride, xf, d[y]);
#pragma unroll
                    for (int x = 0; x < 8; x++) d[y][x] = interp_finish<DEPTH>(d[y][x], 0);
                }
            }
            else if (!xf)
            {
                me_vcol4<P>(r - 3 * (ptrdiff_t)c.rstride, c.rstride, yf, d);
#pragma unroll
                for (int y = 0; y < 4; y++)
#pragma unroll
                    for (int x = 0; x < 8; x++) d[y][x] = interp_finish<DEPTH>(d[y][x], 0);
            }
            else
            {
                me_vmid4(mid + row * c.w + seg * 8, c.w, yf, d);
#pragma unroll
                for (int y = 0; y < 4; y++)
#pragma unroll
                    for (int x = 0; x < 8; x++) d[y][x] = interp_finish<DEPTH>(d[y][x], 2);
            }
#pragma unroll
            for (int y = 0; y < 4; y++)
            {
                int fv[8];
                me_load_fenc<P, 8>(c, c.fenc + (ptrdiff_t)(y0 + row + y) * c.fstride + seg * 8, fv);
#pragma unroll
                for (int x = 0; x < 8; x++) d[y][x] = fv[x] - d[y][x];
            }
            int part = 0;
            if (!satd)
            {
#pragma unroll
                for (int y = 0; y < 4; y++)
#pragma unroll
                    for (int x = 0; x < 8; x++) part += abs(d[y][x]);
            }
            else
            {   // one 8x4 tile (pixel.cpp:239-261): two 4x4 Hadamards, halved together
#pragma unroll
                for (int y = 0; y < 4; y++) { had4(d[y][0], d[y][1], d[y][2], d[y][3]); had4(d[y][4], d[y][5], d[y][6], d[y][7]); }
#pragma unroll
                for (int x = 0; x < 8; x++)
                {
                    had4(d[0][x], d[1][x], d[2][x], d[3][x]);
                    part += abs(d[0][x]) + abs(d[1][x]) + abs(d[2][x]) + abs(d[3][x]);
                }
                part >>= 1;
            }
            acc += part;
        }
    }
    return warp_sum(acc);
}

template <typename P, bool PL = false>
__device__ __forceinline__ int me_subpel_multi_small(const MeCtx<P>& c, int n, int qx, int qy, bool satd)
{
    return c.w >= 8 ? me_subpel_small_t<P, 8, PL>(c, n, qx, qy, satd) : me_subpel_small_t<P, 4, PL>(c, n, qx, qy, satd);
}

// out-of-line copy for the cold multi-site users (pre-checks, lowres band cost)
template <typename P>
__device__ __noinline__ int me_subpel_compare(const MeCtx<P>& c, int qx, int qy, bool satd) { return me_subpel_compare_t(c, qx, qy, satd); }
template <typename P>
__device__ __noinline__ int me_band_cost_ni(const MeCtx<P>& c, int y0, int rows, bool satd) { return me_band_cost(c, y0, rows, satd); }
// subpelCompare of ONE candidate out of the phase planes (AMP sizes): the full-pel compare of its phase plane
template <typename P>
__device__ __noinline__ int me_subpel_compare_pl(const MeCtx<P>& c, int qx, int qy, bool satd)
{
    const P* r = me_qpel_ptr(c, qx, qy);
    if (!satd) return me_sad_direct(c, r);
    return warp_satd(c.fenc, c.fstride, r, c.rstride, c.w, c.h, c.lane);
}

// PU classes of the sub-pel stage: 0 = small (pow2, w and h <= 16: four candidates at a time through
// me_subpel_multi_small), 1 = everything else (one candidate at a time, banded).  CLS = -1 compiles both.
template <typename P>
__device__ __forceinline__ int me_subpel_class(const MeCtx<P>& c) { return (c.pow2 && c.w <= 16 && c.h <= 16) ? 0 : 1; }

// distortion of up to 8 sub-pel candidates, lane i (< n) owns candidate i; result in lane i.  PL: read from the phase planes.
template <typename P, int CLS, bool PL = false>
__device__ __forceinline__ int me_subpel_batch(const MeCtx<P>& c, int n, int qx, int qy, bool satd)
{
    int out = 0;
    if (CLS == 0 || (CLS < 0 && me_subpel_class(c) == 0))
    {
        for (int base = 0; base < n; base += 4)
        {
            const int src = min(base + (c.lane & 3), n - 1);
            const int bqx = __shfl_sync(0xffffffffu, qx, src), bqy = __shfl_sync(0xffffffffu, qy, src);
            int v = me_subpel_multi_small<P, PL>(c, min(4, n - base), bqx, bqy, satd);
            v = __shfl_sync(0xffffffffu, v, (c.lane - base) & 3);
            if (c.lane >= base && c.lane < base + 4) out = v;
        }
    }
    else
    {
        for (int k = 0; k < n; k++)
        {
            const int kqx = __shfl_sync(0xffffffffu, qx, k), kqy = __shfl_sync(0xffffffffu, qy, k);
            int v = c.pow2 ? me_subpel_big<P, PL>(c, kqx, kqy, satd)
                           : PL ? me_subpel_compare_pl(c, kqx, kqy, satd) : me_subpel_compare(c, kqx, kqy, satd);      // AMP sizes: generic, out of line
            if (c.lane == k) out = v;
        }
    }
    return out;
}

// lowresQPelCost (lowres.h:94-120): qpel = rounded average of the two nearest hpel planes; 8x8 blocks
template <typename P>
__device__ __noinline__ int me_lowres_cost(const MeCtx<P>& c, int qx, int qy, bool satd)
{
    if ((qx | qy) & 1)
    {
        int ha = (qy & 2) | ((qx & 2) >> 1);
        const P* a = c.ref[ha] + (qx >> 2) + (ptrdiff_t)(qy >> 2) * c.rstride;
        int rx = qx + (qx & 1), ry = qy + (qy & 1);
        int hb = (ry & 2) | ((rx & 2) >> 1);
        const P* b = c.ref[hb] + (rx >> 2) + (ptrdiff_t)(ry >> 2) * c.rstride;
        __syncwarp();
        for (int i = c.lane; i < 64; i += 32)
        {
            int y = i >> 3, x = i & 7;
            c.sm->pred[y * 64 + x] = (uint16_t)(((int)a[(ptrdiff_t)y * c.rstride + x] + (int)b[(ptrdiff_t)y * c.rstride + x] + 1) >> 1);
        }
        __syncwarp();
        return warp_sum(me_band_cost_ni(c, 0, c.h, satd));
    }
    int hp = (qy & 2) | ((qx & 2) >> 1);
    const P* r = c.ref[hp] + (qx >> 2) + (ptrdiff_t)(qy >> 2) * c.rstride;
    if (!satd) return me_sad_direct(c, r);
    return warp_satd(c.fenc, c.fstride, r, c.rstride, c.w, c.h, c.lane);
}

// SATD partial of one row segment: horizontal 4-point Hadamards in registers, vertical ones over the 4 lanes of a
// tile; returns the halved tile sum in the tile's first lane (0 elsewhere)
template <int NPX>
__device__ __forceinline__ int me_seg_satd(int (&d)[NPX], int lane)
{
#pragma unroll
    for (int x = 0; x < NPX; x += 4) had4(d[x], d[x + 1], d[x + 2], d[x + 3]);
#pragma unroll
    for (int st = 1; st <= 2; st <<= 1)
    {
        const bool up = (lane & st) != 0;
#pragma unroll
        for (int x = 0; x < NPX; x++)
        {
            const int o = __shfl_xor_sync(0xffffffffu, d[x], st);
            d[x] = up ? o - d[x] : o + d[x];
        }
    }
    int part = 0;
#pragma unroll
    for (int x = 0; x < NPX; x++) part += abs(d[x]);
    part += __shfl_xor_sync(0xffffffffu, part, 1);
    part += __shfl_xor_sync(0xffffffffu, part, 2);
    return (lane & 3) ? 0 : (part >> 1);                 // one 8x4 (4x4) tile per 4 lanes, halved per tile
}

// 8 pixels of a reference row at any byte phase
template <typename P>
__device__ __forceinline__ void me_load_row8(const P* __restrict__ p, int (&v)[8])
{
    if (sizeof(P) == 1)
    {
        const uintptr_t a = (uintptr_t)p;
        const uint32_t* ap = (const uint32_t*)(a & ~(uintptr_t)3);
        const unsigned sh = ((unsigned)a & 3u) * 8u;
        const uint32_t w0 = __ldg(ap), w1 = __ldg(ap + 1), w2 = sh ? __ldg(ap + 2) : 0u;
        const uint32_t x0 = __funnelshift_r(w0, w1, sh), x1 = __funnelshift_r(w1, w2, sh);
#pragma unroll
        for (int k = 0; k < 4; k++) { v[k] = (int)((x0 >> (8 * k)) & 255u); v[4 + k] = (int)((x1 >> (8 * k)) & 255u); }
    }
    else
    {
#pragma unroll
        for (int k = 0; k < 8; k++) v[k] = (int)__ldg(p + k);
    }
}

// lowresQPelCost (lowres.h:94-120) of up to 4 candidates of an 8x8 lowres CU at once: 8 lanes per candidate, one
// row each; the row of the prediction (one half-pel plane, or the rounded average of the two nearest for odd
// quarter-pel positions) stays in registers, SATD = two 8x4 tiles through the shuffle butterflies.  Lane i (< n)
// gets candidate i's distortion.  Same arithmetic as me_lowres_cost.
template <typename P>
__device__ __forceinline__ int me_lowres_multi(const MeCtx<P>& c, int n, int qx, int qy, bool satd)
{
    const int lane = c.lane, slot = lane >> 3, row = lane & 7;
    const int cand = min(slot, n - 1);
    const int mqx = __shfl_sync(0xffffffffu, qx, cand), mqy = __shfl_sync(0xffffffffu, qy, cand);
    int d[8];
    {
        const int ha = (mqy & 2) | ((mqx & 2) >> 1);
        const P* pa = ha == 0 ? c.ref[0] : ha == 1 ? c.ref[1] : ha == 2 ? c.ref[2] : c.ref[3];
        int a[8];
        me_load_row8<P>(pa + (mqx >> 2) + (ptrdiff_t)((mqy >> 2) + row) * c.rstride, a);
        if ((mqx | mqy) & 1)
        {
            const int rx = mqx + (mqx & 1), ry = mqy + (mqy & 1);
            const int hb = (ry & 2) | ((rx & 2) >> 1);
            const P* pb = hb == 0 ? c.ref[0] : hb == 1 ? c.ref[1] : hb == 2 ? c.ref[2] : c.ref[3];
            int b[8];
            me_load_row8<P>(pb + (rx >> 2) + (ptrdiff_t)((ry >> 2) + row) * c.rstride, b);
#pragma unroll
            for (int x = 0; x < 8; x++) a[x] = (a[x] + b[x] + 1) >> 1;
        }
        int fv[8];
        me_load_fenc<P, 8>(c, c.fenc + (ptrdiff_t)row * c.fstride, fv);
#pragma unroll
        for (int x = 0; x < 8; x++) d[x] = slot < n ? fv[x] - a[x] : 0;
    }
    int part = 0;
    if (!satd)
    {
#pragma unroll
        for (int x = 0; x < 8; x++) part += abs(d[x]);
        part += __shfl_xor_sync(0xffffffffu, part, 1);
        part += __shfl_xor_sync(0xffffffffu, part, 2);
    }
    else part = me_seg_satd<8>(d, lane);
    part += __shfl_xor_sync(0xffffffffu, part, 4);
    return __shfl_sync(0xffffffffu, part, (lane << 3) & 31);
}

// distortion of up to 8 lowres candidates, lane i (< n) owns candidate i
template <typename P>
__device__ __forceinline__ int me_lowres_batch(const MeCtx<P>& c, int n, int qx, int qy, bool satd)
{
    int out = 0;
    for (int base = 0; base < n; base += 4)
    {
        const int src = min(base + (c.lane & 3), n - 1);
        const int bqx = __shfl_sync(0xffffffffu, qx, src), bqy = __shfl_sync(0xffffffffu, qy, src);
        int v = me_lowres_multi(c, min(4, n - base), bqx, bqy, satd);
        v = __shfl_sync(0xffffffffu, v, (c.lane - base) & 3);
        if (c.lane >= base && c.lane < base + 4) out = v;
    }
    return out;
}

template <typename P>
__device__ __forceinline__ int me_qpel_cost(const MeCtx<P>& c, int qx, int qy, bool satd)
{
    return c.lowres ? me_lowres_cost(c, qx, qy, satd) : me_subpel_compare(c, qx, qy, satd);
}

template <typename P>
__device__ __forceinline__ int me_cost_fpel(const MeCtx<P>& c, int x, int y)
{
    return me_sad_direct(c, c.ref[0] + x + (ptrdiff_t)y * c.rstride) + me_mvcost(c, x * 4, y * 4);
}

struct MeStar { int bx, by, bcost, point, dist; };

// shared-memory search window context (me_window.cuh): its evaluation sites are overloads of the same names
template <typename P> struct MeWin;
template <typename P> __device__ __forceinline__ int me_eval_points(const MeWin<P>& c, int n, int px, int py, bool x8);
template <typename P> __device__ __forceinline__ void me_raster(const MeWin<P>& c, MeStar& s);

// Fold a burst in the reference's order.  The sequential `if (cost < bcost)` chain keeps the EARLIEST
// candidate among those reaching the minimum, so it equals one arg-min with ties to the lowest index:
// pack (cost << 5 | index) and take a single warp min (REDUX.MIN).  Costs stay below 2^26.
__device__ __forceinline__ int me_argmin(int n, int cost, int lane)
{
    unsigned key = (lane < n) ? (((unsigned)cost << 5) | (unsigned)lane) : 0xffffffffu;
    return (int)__reduce_min_sync(0xffffffffu, key);
}
__device__ __forceinline__ void me_fold(MeStar& s, int n, int cost, int px, int py, int point, int dist)
{
    if (n <= 0) return;
    const int lane = threadIdx.x & 31;
    const unsigned key = (unsigned)me_argmin(n, cost, lane);
    const int best = (int)(key >> 5), i = (int)(key & 31);
    if (best < s.bcost)
    {
        s.bcost = best;
        s.bx = __shfl_sync(0xffffffffu, px, i); s.by = __shfl_sync(0xffffffffu, py, i);
        s.point = __shfl_sync(0xffffffffu, point, i); s.dist = __shfl_sync(0xffffffffu, dist, i);
    }
}

// StarPatternSearch (motion.cpp:362-604).  Each distance level is one burst; candidate order inside
// a level is the reference's (its x4 fast path and its bounds-checked path visit the same points in
// the same order), out-of-range candidates are dropped before evaluation.
// Candidate k of star level `mylvl` around (ox, oy) (motion.cpp:362-604; the order inside a level is the reference's):
// levels 0 = distance 1 (4 points), 1..3 = distances 2, 4, 8 (8 points), 4.. = distances 16, 32, ... (16 points).
__device__ __forceinline__ void me_star_point(int mylvl, int k, int ox, int oy, int& px, int& py, int& point, int& dist)
{
    const int d = mylvl < 4 ? (1 << mylvl) : (16 << (mylvl - 4));
    if (mylvl == 0)
    {
        // dist 1: top(2) left(4) right(5) bottom(7)
        px = ox + (k == 1 ? -1 : k == 2 ? 1 : 0); py = oy + (k == 0 ? -1 : k == 3 ? 1 : 0);
        point = k == 0 ? 2 : k == 1 ? 4 : k == 2 ? 5 : 7; dist = 1;
    }
    else if (mylvl < 4)
    {
        // order: 2(top) 1 3 4(left) 5(right) 6 8 7(bottom); half-distance points need both their checks
        const int h2 = d >> 1, kk = k & 7;
        const int dx = kk == 0 ? 0 : kk == 1 ? -1 : kk == 2 ? 1 : kk == 3 ? -2 : kk == 4 ? 2 : kk == 5 ? -1 : kk == 6 ? 1 : 0;
        const int dy = kk == 0 ? -2 : kk < 3 ? -1 : kk < 5 ? 0 : kk < 7 ? 1 : 2;
        px = ox + dx * h2; py = oy + dy * h2;
        point = kk == 0 ? 2 : kk == 1 ? 1 : kk == 2 ? 3 : kk == 3 ? 4 : kk == 4 ? 5 : kk == 5 ? 6 : kk == 6 ? 8 : 7;
        dist = (kk == 1 || kk == 2 || kk == 5 || kk == 6) ? h2 : d;
    }
    else
    {
        // order: top, left, right, bottom, then j = 1..3: (xl,yt) (xr,yt) (xl,yb) (xr,yb)
        const int q = d >> 2, kk = k & 15;
        if (kk < 4) { px = ox + (kk == 1 ? -d : kk == 2 ? d : 0); py = oy + (kk == 0 ? -d : kk == 3 ? d : 0); }
        else
        {
            const int jj = ((kk - 4) >> 2) + 1, m = (kk - 4) & 3;
            px = ox + ((m & 1) ? q * jj : -q * jj);
            py = (m & 2) ? (oy + d - q * jj) : (oy - d + q * jj);
        }
        point = 0; dist = d;
    }
}

// Hooks of the shared-memory-window search (me_window.cuh): the first star round of a 16x16 cell's PUs that start at the
// same point reads its candidates' SADs from a table computed once per cell.  Global-memory contexts never have one.
template <typename P> __device__ __forceinline__ bool me_star_cached(const MeCtx<P>&) { return false; }
template <typename P> __device__ __forceinline__ int me_star_lookup(const MeCtx<P>&, int, int, int, int) { return 0; }
template <typename P> struct MeWinCell;
template <typename P> __device__ __forceinline__ bool me_star_cached(const MeWin<P>&);
template <typename P> __device__ __forceinline__ int me_star_lookup(const MeWin<P>&, int, int, int, int);
template <typename P> __device__ __forceinline__ bool me_star_cached(const MeWinCell<P>& c);
template <typename P> __device__ __forceinline__ int me_star_lookup(const MeWinCell<P>& c, int mylvl, int k, int px, int py);

template <typename CTX>
__device__ __forceinline__ void me_star_pattern(const CTX& c, MeStar& s, int earlyExitIters, int merange, bool first = false)
{
    // Levels: 0 = distance 1 (4 points), 1..3 = distances 2, 4, 8 (8 points), 4.. = distances 16, 32, ... <= merange
    // (16 points).  Every level's points depend only on the start position, so levels can be evaluated ahead of the
    // early-exit decision without changing it: for small PUs (<= 64 words, where the per-burst bookkeeping costs more
    // than the SADs) levels 0-3 form ONE burst of 28 candidates and the far levels go two per burst; the decisions
    // are then replayed level by level with a masked arg-min.  Large PUs keep one level per burst (no wasted SADs).
    // One loop, one evaluation site (the SAD core is inlined).
    const int ox = s.bx, oy = s.by, lane = c.lane;
    const bool spec = c.pow2 && c.nw <= 64;
    int rounds = 0, lvl0 = 0;
    for (;;)
    {
        const int lvl1 = !spec ? lvl0 + 1 : (lvl0 == 0 ? 4 : lvl0 + 2);
        int mylvl, k;
        if (!spec)          { mylvl = lvl0; k = lane; }
        else if (lvl0 == 0) { mylvl = lane < 4 ? 0 : 1 + ((lane - 4) >> 3); k = lane < 4 ? lane : (lane - 4) & 7; }
        else                { mylvl = lvl0 + (lane >> 4); k = lane & 15; }
        const int d = mylvl < 4 ? (1 << mylvl) : (16 << (mylvl - 4));
        const int cnt = mylvl == 0 ? 4 : mylvl < 4 ? 8 : 16;
        int px, py, point, dist;
        me_star_point(mylvl, k, ox, oy, px, py, point, dist);
        const bool valid = mylvl < lvl1 && k < cnt && !(mylvl >= 4 && d > merange) &&
                           px >= c.minx && px <= c.maxx && py >= c.miny && py <= c.maxy;
        // idle lanes evaluate an in-range position (the centre clamped into the search range: the start point can lie outside
        // it in x when MV 0 won the pre-checks, motion.cpp:806-813) and are masked out
        if (!valid) { px = min(max(ox, c.minx), c.maxx); py = min(max(oy, c.miny), c.maxy); }
        const int n = spec ? (lvl0 == 0 ? 28 : 32) : (lvl0 == 0 ? 4 : lvl0 < 4 ? 8 : 16);
        // the first round of a cell's PUs that share the start point: SADs out of the cell's star table (me_window.cuh)
        const int cost = (first && me_star_cached(c)) ? (valid ? me_star_lookup(c, mylvl, k, px, py) : 0x7fffffff)
                                                      : me_eval_points(c, n, px, py, false);
        for (int l = lvl0; l < lvl1; l++)
        {
            if (l >= 4 && (16 << (l - 4)) > merange) return;
            const int saved = s.bcost;
            const unsigned key = (valid && mylvl == l) ? (((unsigned)cost << 5) | (unsigned)lane) : 0xffffffffu;
            const unsigned m = __reduce_min_sync(0xffffffffu, key);
            if (m != 0xffffffffu && (int)(m >> 5) < s.bcost)
            {
                const int src = (int)(m & 31);
                s.bcost = (int)(m >> 5);
                s.bx = __shfl_sync(0xffffffffu, px, src); s.by = __shfl_sync(0xffffffffu, py, src);
                s.point = __shfl_sync(0xffffffffu, point, src); s.dist = __shfl_sync(0xffffffffu, dist, src);
            }
            if (s.bcost < saved) rounds = 0;
            else if (++rounds >= earlyExitIters) return;
        }
        lvl0 = lvl1;
        if (lvl0 >= 4 && (16 << (lvl0 - 4)) > merange) return;
    }
}

__constant__ int8_t c_hex2[8][2]    = { {-1,-2}, {-2,0}, {-1,2}, {1,2}, {2,0}, {1,-2}, {-1,-2}, {-2,0} };
__constant__ uint8_t c_mod6m1[8]    = { 5, 0, 1, 2, 3, 4, 5, 0 };
__constant__ int8_t c_square1[9][2] = { {0,0}, {0,-1}, {0,1}, {-1,0}, {1,0}, {-1,-1}, {-1,1}, {1,-1}, {1,1} };
__constant__ int8_t c_star_off[16][2] = { {-1,0},{0,-1}, {-1,-1},{1,-1}, {-1,0},{1,0}, {-1,1},{-1,-1},
                                          {1,-1},{1,1}, {-1,0},{0,1}, {-1,1},{1,1}, {1,0},{0,1} };
// motion.cpp:48-58 {hpel_iters, hpel_dirs, qpel_iters, qpel_dirs, hpel_satd}
__constant__ int8_t c_workload[8][5] = { {1,4,0,4,0}, {1,4,1,4,0}, {1,4,1,4,1}, {2,4,1,4,1}, {2,4,2,4,1}, {1,8,1,8,1}, {2,8,1,8,1}, {2,8,2,8,1} };

// ---- chroma-SATD term of subpelCompare (motion.cpp:1601-1661), 4:2:0 -----------------------------------------
// With bChromaSATD (subme > 2 and a chroma block that is a multiple of 4x4: motion.cpp:204-212) EVERY subpelCompare
// adds chromaSatd(Cb) + chromaSatd(Cr) of the chroma block predicted at the eighth-pel vector (mvx = qmv.x for
// 4:2:0): filter_hpp / filter_vpp / filter_hps(rowExt) + filter_vsp with the 4-tap filter.
struct MeChromaArgs                        // device pointers; the chroma pixel of luma (x, y) is at (y >> 1) * cstride + (x >> 1)
{
    const void* fencCb; const void* fencCr;
    const void* const* refCb; const void* const* refCr;      // device arrays of plane pointers, indexed by job.ref
    int cstride;
};

// per-job chroma context (kept out of MeCtx so that the luma-only kernels are not touched by it)
template <typename P>
struct MeChromaCtx
{
    bool on;                               // MotionEstimate::bChromaSATD of this job (motion.cpp:204-212)
    const P* fcb; const P* fcr;            // source Cb / Cr at the PU's chroma origin
    const P* rcb; const P* rcr;            // reference Cb / Cr at the PU's chroma origin
    int cstride;
};

template <typename P>
__device__ __forceinline__ void me_set_chroma(MeChromaCtx<P>& cc, const MeCtx<P>& c, const x265cu_me_job& j, const MeChromaArgs& a, int fstride)
{
    cc.on = !c.lowres && j.subme > 2 && !(c.w & 7) && !(c.h & 7);
    const int py = j.offset / fstride, px = j.offset - py * fstride;
    const ptrdiff_t coff = (ptrdiff_t)(py >> 1) * a.cstride + (px >> 1);
    cc.cstride = a.cstride;
    cc.fcb = (const P*)a.fencCb + coff; cc.fcr = (const P*)a.fencCr + coff;
    cc.rcb = ((const P* const*)a.refCb)[j.ref] + coff; cc.rcr = ((const P* const*)a.refCr)[j.ref] + coff;
}

// N consecutive pixels starting at p (any alignment) as ints: aligned 32-bit loads + funnel shifts instead of N scalar
// loads (the chroma tiles are 4 wide + 3 taps: seven byte loads per row cost seven L1 requests, three words cost three).
// Reads up to 3 bytes before / 4 bytes after the span inside the same words (the planes have margins).
template <typename P, int N>
__device__ __forceinline__ void me_ld_px(const P* __restrict__ p, int (&v)[N])
{
    constexpr int NB = N * (int)sizeof(P), NWD = (NB + 3) / 4;                 // payload bytes / words after alignment
    const uintptr_t a = (uintptr_t)p;
    const uint32_t* ap = (const uint32_t*)(a & ~(uintptr_t)3);
    const unsigned sh = ((unsigned)a & 3u) * 8u;
    uint32_t w[NWD + 1], x[NWD];
#pragma unroll
    for (int k = 0; k <= NWD; k++) w[k] = __ldg(ap + k);
#pragma unroll
    for (int k = 0; k < NWD; k++) x[k] = __funnelshift_r(w[k], w[k + 1], sh);
#pragma unroll
    for (int i = 0; i < N; i++)
        v[i] = sizeof(P) == 1 ? (int)((x[i >> 2] >> (8 * (i & 3))) & 255u) : (int)((x[i >> 1] >> (16 * (i & 1))) & 65535u);
}

// the 4-tap chroma filters as packed signed bytes (DP4A / DP2A operand): all taps are within [-6, 64].  In GLOBAL memory:
// the lanes of a pass look up different phases, which a constant-bank access would serialise.
__device__ const uint32_t d_chromaTaps4[8] = {
    0x00004000u, 0xfe0a3afeu, 0xfe1036fcu, 0xfc1c2efau, 0xfc2424fcu, 0xfa2e1cfcu, 0xfc3610feu, 0xfe3a0afeu };

// un-normalised 4-tap horizontal sums of the 4 outputs whose support is the 7 pixels starting at p (any alignment):
// aligned words + funnel shifts, then one DP4A (8-bit) / two DP2A (16-bit) per output instead of four IMADs and the
// per-pixel extraction.  Reads up to 3 bytes before / 5 bytes after the span inside the same words (plane margins).
template <typename P>
__device__ __forceinline__ void me_chroma_hsum4(const P* __restrict__ p, uint32_t taps, int (&s)[4])
{
    const uintptr_t a = (uintptr_t)p;
    const uint32_t* ap = (const uint32_t*)(a & ~(uintptr_t)3);
    const unsigned sh = ((unsigned)a & 3u) * 8u;
    if (sizeof(P) == 1)
    {
        const uint32_t w0 = __ldg(ap), w1 = __ldg(ap + 1), w2 = __ldg(ap + 2);
        const uint32_t x0 = __funnelshift_r(w0, w1, sh), x1 = __funnelshift_r(w1, w2, sh);
        s[0] = dp4a_us(x0, taps, 0);
        s[1] = dp4a_us(__funnelshift_r(x0, x1, 8), taps, 0);
        s[2] = dp4a_us(__funnelshift_r(x0, x1, 16), taps, 0);
        s[3] = dp4a_us(__funnelshift_r(x0, x1, 24), taps, 0);
    }
    else
    {
        uint32_t w[5], x[4];
#pragma unroll
        for (int k = 0; k < 5; k++) w[k] = __ldg(ap + k);
#pragma unroll
        for (int k = 0; k < 4; k++) x[k] = __funnelshift_r(w[k], w[k + 1], sh);
        const uint32_t p1 = __funnelshift_r(x[0], x[1], 16), p3 = __funnelshift_r(x[1], x[2], 16), p5 = __funnelshift_r(x[2], x[3], 16);
        s[0] = dp2a_hi_ss(x[1], taps, dp2a_lo_ss(x[0], taps, 0));
        s[1] = dp2a_hi_ss(p3, taps, dp2a_lo_ss(p1, taps, 0));
        s[2] = dp2a_hi_ss(x[2], taps, dp2a_lo_ss(x[1], taps, 0));
        s[3] = dp2a_hi_ss(p5, taps, dp2a_lo_ss(p3, taps, 0));
    }
}

// un-normalised 4x4 Hadamard abs-sum of (source chroma block - predicted chroma block).  One lane, registers only;
// out of line (one copy per kernel: the ME kernels are instruction-cache sensitive).
// ONE code path for all fractional phases: the separable form filter_hps(rowExt) -> filter_vsp of the reference's hv case
// (ipfilter.cpp:120-162, 241-282) with the identity taps {0, 64, 0, 0} for a zero phase reproduces the direct forms exactly:
//   yf == 0 is excluded below only for 10-bit horizontal-only phases, where hps drops two bits that hpp keeps;
//   xf == 0: mid = 64 p - 8192 (8-bit) / 16 p - 8192 (10-bit) is exact, so vsp gives (sum(c p) + 32) >> 6 = filter_vpp;
//   xf == yf == 0: the pixel itself.
// Lanes of a pass hold candidates of different phases: a single path means no divergence and a small body (the kernels
// with this term ran at a 60 % instruction-cache hit rate with the four-way version).
template <typename P>
__device__ __noinline__ int me_chroma_had4x4(const P* __restrict__ f, const P* __restrict__ r, int stride, int xf, int yf)
{
    constexpr int DEPTH = PixTraits<P>::depth;
    int m[4][4];
    if (DEPTH != 8 && xf && !yf)
    {   // 10-bit horizontal only: filter_hpp directly
        const uint32_t th = __ldg(&d_chromaTaps4[xf]);
#pragma unroll
        for (int y = 0; y < 4; y++)
        {
            int hs[4];
            me_chroma_hsum4<P>(r + y * stride - 1, th, hs);
#pragma unroll
            for (int x = 0; x < 4; x++) m[y][x] = interp_finish<DEPTH>(hs[x], 0);
        }
    }
    else
    {
        const uint32_t th = __ldg(&d_chromaTaps4[xf]);
        const uint32_t tv = __ldg(&d_chromaTaps4[yf]);
        const int v0 = (int)(int8_t)tv, v1 = (int)(int8_t)(tv >> 8), v2 = (int)(int8_t)(tv >> 16), v3 = (int)tv >> 24;
        int mid[7][4];                     // filter_hps with isRowExt: rows -1 .. +5 of the block (ipfilter.cpp:120-162)
#pragma unroll
        for (int k = 0; k < 7; k++)
        {
            int hs[4];
            me_chroma_hsum4<P>(r + (k - 1) * stride - 1, th, hs);
#pragma unroll
            for (int x = 0; x < 4; x++) mid[k][x] = interp_finish<DEPTH>(hs[x], 1);
        }
#pragma unroll
        for (int y = 0; y < 4; y++)
#pragma unroll
            for (int x = 0; x < 4; x++)
                m[y][x] = interp_finish<DEPTH>(v0 * mid[y][x] + v1 * mid[y + 1][x] + v2 * mid[y + 2][x] + v3 * mid[y + 3][x], 2);
    }
#pragma unroll
    for (int y = 0; y < 4; y++)
    {
        int fv[4];
        me_ld_px<P, 4>(f + y * stride, fv);
#pragma unroll
        for (int x = 0; x < 4; x++) m[y][x] = fv[x] - m[y][x];
        had4(m[y][0], m[y][1], m[y][2], m[y][3]);
    }
    int acc = 0;
#pragma unroll
    for (int x = 0; x < 4; x++)
    {
        had4(m[0][x], m[1][x], m[2][x], m[3][x]);
        acc += abs(m[0][x]) + abs(m[1][x]) + abs(m[2][x]) + abs(m[3][x]);
    }
    return acc;
}

// position of the (n + 1)-th set bit of `mask` (n < popc(mask)): five halving steps on population counts (__fns is a
// long software loop: it was 17 % of the instructions of the chroma kernels)
__device__ __forceinline__ int me_nth_set_bit(unsigned mask, int n)
{
    int pos = 0;
#pragma unroll
    for (int w = 16; w >= 1; w >>= 1)
    {
        const int c = __popc(mask & ((1u << w) - 1u));
        if (n >= c) { n -= c; mask >>= w; pos += w; }
    }
    return pos;
}

// un-normalised 4-tap horizontal sum of the four pixels starting at p (any alignment): aligned words, funnel shifts and
// one DP4A (8-bit) / two DP2A (16-bit) -- exact in int32
template <typename P>
__device__ __forceinline__ int me_chroma_hsum(const P* __restrict__ p, uint32_t taps)
{
    const uintptr_t a = (uintptr_t)p;
    const uint32_t* ap = (const uint32_t*)(a & ~(uintptr_t)3);
    const unsigned sh = ((unsigned)a & 3u) * 8u;
    if (sizeof(P) == 1)
    {
        const uint32_t w0 = __ldg(ap), w1 = __ldg(ap + 1);
        return dp4a_us(__funnelshift_r(w0, w1, sh), taps, 0);
    }
    else
    {
        const uint32_t w0 = __ldg(ap), w1 = __ldg(ap + 1), w2 = __ldg(ap + 2);
        return dp2a_hi_ss(__funnelshift_r(w1, w2, sh), taps, dp2a_lo_ss(__funnelshift_r(w0, w1, sh), taps, 0));
    }
}

// Cb + Cr chroma SATD of the candidates of a burst: lane k (k < n, bit k of `need` set) receives candidate k's cost.
// chromaSatd is the luma SATD primitive of the chroma-sized block (primitives.cpp:139-158): 8x4 tiles when the chroma
// width is a multiple of 8, else 4x4 tiles, each tile halved on its own (pixel.cpp:210-297, 1131-1155).
//
// CLS 1 (large / non power-of-two PUs): work items = (needed candidate, plane, tile), one lane per tile, candidate-major,
// 32 at a time (a 32x32 PU has 16 tiles per candidate: the warp is full); per-candidate sums are one REDUX each.
template <typename P>
__device__ __forceinline__ int me_chroma_batch_tiles(const MeCtx<P>& c, const MeChromaCtx<P>& cc, int n, int qx, int qy, unsigned need)
{
    const int cw = c.w >> 1, chh = c.h >> 1;
    const int tw = (cw & 7) ? 4 : 8;
    const int tpr = cw / tw, nt = tpr * (chh >> 2);                 // tiles per row / per plane
    const int ipc = 2 * nt;                                        // items per candidate
    if (n < 32) need &= (1u << n) - 1u;
    const int nneed = __popc(need);
    const int total = nneed * ipc;
    int out = 0;
    for (int base = 0; base < total; base += 32)
    {
        const int it = base + c.lane;
        const bool live = it < total;
        const int ci = live ? it / ipc : 0;
        const int rem = it - ci * ipc;
        const int k = need == (nneed >= 32 ? 0xffffffffu : ((1u << nneed) - 1u)) ? ci : me_nth_set_bit(need, ci);   // the ci-th needed candidate
        const int kqx = __shfl_sync(0xffffffffu, qx, k & 31), kqy = __shfl_sync(0xffffffffu, qy, k & 31);
        int v = 0;
        if (live)
        {
            const bool cr = rem >= nt;
            const int tt = cr ? rem - nt : rem;
            const int ty = tt / tpr, tx = tt - ty * tpr;
            const int xf = kqx & 7, yf = kqy & 7;
            const ptrdiff_t roff = (kqx >> 3) + (ptrdiff_t)(kqy >> 3) * cc.cstride;
            const ptrdiff_t o = (ptrdiff_t)(ty * 4) * cc.cstride + tx * tw;
            const P* f = (cr ? cc.fcr : cc.fcb) + o;
            const P* r = (cr ? cc.rcr : cc.rcb) + o + roff;
            v = me_chroma_had4x4<P>(f, r, cc.cstride, xf, yf);
            if (tw == 8) v += me_chroma_had4x4<P>(f + 4, r + 4, cc.cstride, xf, yf);
            v >>= 1;
        }
        __syncwarp();
        // candidates present in this chunk: ci in [base / ipc, (base + 31) / ipc]
        const int c0 = base / ipc, c1 = min(nneed - 1, (base + 31) / ipc);
        for (int q = c0; q <= c1; q++)
        {
            const int tot = __reduce_add_sync(0xffffffffu, (live && ci == q) ? v : 0);
            const int kq = me_nth_set_bit(need, q);
            if (c.lane == kq) out += tot;
        }
    }
    return out;
}

// CLS 0 (8x8, 16x8, 8x16, 16x16 PUs: chroma blocks of 1, 2, 2, 4 4x4 tiles per plane): a refinement round has 4-8
// candidates of 2-8 tiles, so one lane per tile leaves most of the warp idle while it issues the whole 600-instruction
// tile function.  Here FOUR lanes share a 4x4 tile, one COLUMN each: a lane's 7 horizontal sums (rows -1 .. +5 of its
// column, one DP4A each) are exactly what its 4 outputs need -- no redundant filtering --, the vertical Hadamard is in-lane and
// the horizontal one two shuffle butterflies.  Lane-items per candidate = 8 / 16 / 32 (powers of two: shifts, no
// divisions; a candidate never straddles a pass), so tile and candidate sums are xor butterflies too.  An 8x8 PU's round
// of 4 candidates is ONE pass of ~200 instructions with all 32 lanes busy (was: 8 lanes x 600); the body is 1/4 the size.
// One code path for all fractional phases as in me_chroma_had4x4 (identity taps for a zero phase; 10-bit
// horizontal-only phases take filter_hpp's rounding by a select).
template <typename P>
__device__ __forceinline__ int me_chroma_batch_cols(const MeCtx<P>& c, const MeChromaCtx<P>& cc, int n, int qx, int qy, unsigned need)
{
    constexpr int DEPTH = PixTraits<P>::depth;
    const int lgtpr = c.lgw - 3;                                   // log2(4x4 tiles per chroma row): 0 or 1
    const int lgnt = lgtpr + (31 - __clz(c.h)) - 3;                // log2(4x4 tiles per plane): 0 .. 2
    const int lgipc = lgnt + 3;                                    // log2(lane-items per candidate): 2 planes x tiles x 4 columns
    const int lggs = 2 + lgtpr;                                    // log2(lanes per SATD tile): 4x4 -> 4 lanes, 8x4 -> 8
    if (n < 32) need &= (1u << n) - 1u;
    const int nneed = __popc(need);
    const int total = nneed << lgipc;
    const bool dense = need == (nneed >= 32 ? 0xffffffffu : ((1u << nneed) - 1u));
    const int myq = __popc(need & ((1u << c.lane) - 1u));           // rank of this lane's candidate among the needed ones
    const int col = c.lane & 3;
    const int s1 = (c.lane & 1) ? -1 : 1, s2 = (c.lane & 2) ? -1 : 1;
    int out = 0;
    for (int base = 0; base < total; base += 32)
    {
        const int it = min(base + c.lane, total - 1);              // idle lanes (whole candidates) redo the last item: harmless
        const int ci = it >> lgipc;
        const int t = (it & ((1 << lgipc) - 1)) >> 2;              // tile of the candidate, both planes
        const int k = dense ? ci : me_nth_set_bit(need, ci);
        const int kqx = __shfl_sync(0xffffffffu, qx, k & 31), kqy = __shfl_sync(0xffffffffu, qy, k & 31);
        const bool cr = (t >> lgnt) != 0;
        const int tt = t & ((1 << lgnt) - 1);
        const int ty = tt >> lgtpr, tx = tt & ((1 << lgtpr) - 1);
        const int xf = kqx & 7, yf = kqy & 7;
        const ptrdiff_t o = (ptrdiff_t)(ty * 4) * cc.cstride + tx * 4 + col;
        const P* f = (cr ? cc.fcr : cc.fcb) + o;
        const P* r = (cr ? cc.rcr : cc.rcb) + o + (kqx >> 3) + (ptrdiff_t)(kqy >> 3) * cc.cstride - 1 - cc.cstride;
        const uint32_t th = __ldg(&d_chromaTaps4[xf]);
        const uint32_t tv = __ldg(&d_chromaTaps4[yf]);
        const int v0 = (int)(int8_t)tv, v1 = (int)(int8_t)(tv >> 8), v2 = (int)(int8_t)(tv >> 16), v3 = (int)tv >> 24;
        int S[7];
#pragma unroll
        for (int q = 0; q < 7; q++) S[q] = me_chroma_hsum<P>(r + q * cc.cstride, th);
        int d[4];
#pragma unroll
        for (int y = 0; y < 4; y++)
        {
            const int m = interp_finish<DEPTH>(v0 * interp_finish<DEPTH>(S[y], 1) + v1 * interp_finish<DEPTH>(S[y + 1], 1) +
                                               v2 * interp_finish<DEPTH>(S[y + 2], 1) + v3 * interp_finish<DEPTH>(S[y + 3], 1), 2);
            const int mh = DEPTH != 8 ? interp_finish<DEPTH>(S[y + 1], 0) : 0;      // filter_hpp keeps the two bits hps drops
            d[y] = (int)__ldg(f + y * cc.cstride) - ((DEPTH != 8 && !yf) ? mh : m);
        }
        had4(d[0], d[1], d[2], d[3]);
#pragma unroll
        for (int y = 0; y < 4; y++)
        {
            d[y] = __shfl_xor_sync(0xffffffffu, d[y], 1) + s1 * d[y];
            d[y] = __shfl_xor_sync(0xffffffffu, d[y], 2) + s2 * d[y];
        }
        int v = abs(d[0]) + abs(d[1]) + abs(d[2]) + abs(d[3]);
        v += __shfl_xor_sync(0xffffffffu, v, 1);
        v += __shfl_xor_sync(0xffffffffu, v, 2);
        if (lggs == 3) v += __shfl_xor_sync(0xffffffffu, v, 4);
        v >>= 1;                                                   // every lane of the tile holds its halved SATD
        for (int s = lggs; s < lgipc; s++) v += __shfl_xor_sync(0xffffffffu, v, 1 << s);   // ... and now the candidate's sum
        const int src = (myq << lgipc) - base;
        const int got = __shfl_sync(0xffffffffu, v, src & 31);
        if (src >= 0 && src < 32 && ((need >> c.lane) & 1u)) out += got;
    }
    return out;
}

template <typename P, int CLS>
__device__ __forceinline__ int me_chroma_batch(const MeCtx<P>& c, const MeChromaCtx<P>& cc, int n, int qx, int qy, unsigned need)
{
    if (CLS == 0) return me_chroma_batch_cols<P>(c, cc, n, qx, qy, need);
    return me_chroma_batch_tiles<P>(c, cc, n, qx, qy, need);
}

struct MeState { int bmx, bmy, bcost, bprecost, bestprex, bestprey; };

#define ME_YOK(y) (((y) >= c.miny) & ((y) <= c.maxy))
#define ME_INRANGE(x, y) ((x) >= c.minx && (x) <= c.maxx && (y) >= c.miny && (y) <= c.maxy)

// phase 1 (motion.cpp:771-814): cost at the clipped MVP, at its full-pel rounding, at MV 0 and at the qpel candidates.
// PL: the luma SADs are one burst of full-pel SADs over the quarter-pel phase planes.
template <typename P, int CLS, bool CHROMA = false, bool PL = false>
__device__ __forceinline__ void me_phase1(MeCtx<P>& c, const x265cu_me_job& j, MeState& st, const MeChromaCtx<P>* cc = nullptr)
{

    const int qminx = c.minx * 4, qminy = c.miny * 4, qmaxx = c.maxx * 4, qmaxy = c.maxy * 4;
    // clipped() = min with max first, then max with min (mv.h:100-105)
    const int pmvx = max(min(c.mvpx, qmaxx), qminx), pmvy = max(min(c.mvpy, qmaxy), qminy);
    int bestprex = pmvx, bestprey = pmvy;
    int bprecost, bmx = (pmvx + 2) >> 2, bmy = (pmvy + 2) >> 2, bcost;
    if (c.lowres)
    {
        {
            // lane 0 = clipped MVP (qpel), lane 1 = its full-pel rounding, lane 2 = MV 0: one burst of SADs
            const int l = c.lane;
            const int bqx = l == 0 ? pmvx : l == 1 ? bmx * 4 : 0, bqy = l == 0 ? pmvy : l == 1 ? bmy * 4 : 0;
            const int cost = me_lowres_multi(c, 3, bqx, bqy, false);
            bprecost = __shfl_sync(0xffffffffu, cost, 0);
            bcost = bprecost;
            if ((pmvx & 3) | (pmvy & 3)) bcost = __shfl_sync(0xffffffffu, cost, 1) + me_mvcost(c, bmx * 4, bmy * 4);
            if (pmvx | pmvy)
            {
                const int cz = __shfl_sync(0xffffffffu, cost, 2) + me_mvcost(c, 0, 0);
                if (cz < bcost) { bcost = cz; bmx = 0; bmy = max(min(0, c.maxy), c.miny); }
            }
        }
#pragma unroll
        for (int i = 0; i < 4; i++)                         // static indices keep the job record in registers
        {
            if (i >= j.numCand) break;
            int mx = max(min((int)j.mvc[2 * i], qmaxx), qminx), my = max(min((int)j.mvc[2 * i + 1], qmaxy), qminy);
            if ((mx | my) && !(mx == pmvx && my == pmvy) && !(mx == bestprex && my == bestprey))
            {
                int cost = me_subpel_compare(c, mx, my, false) + me_mvcost(c, mx, my);
                if (cost < bprecost) { bprecost = cost; bestprex = mx; bestprey = my; }
            }
        }
    }
    else
    {
        // All the pre-checks are SADs at independent positions: ONE burst.  Lane 0 = clipped MVP (qpel), lane 1 = its
        // full-pel rounding (only when the MVP is fractional), lane 2 = MV 0 (only when the MVP is not 0), lanes 3.. =
        // the qpel candidates.  The reference skips a candidate equal to the best so far; evaluating it is harmless (its
        // cost equals that best and '<' is strict), so the candidate fold is one arg-min with ties to the earliest.
        const int lane = c.lane, ci = min(max(lane - 3, 0), 3);
        int mvl = 0;                                        // lane k holds mvc[k]: no dynamic indexing of the job record
#pragma unroll
        for (int k = 0; k < 8; k++) mvl = (lane == k) ? (int)j.mvc[k] : mvl;
        const int candx = __shfl_sync(0xffffffffu, mvl, 2 * ci), candy = __shfl_sync(0xffffffffu, mvl, 2 * ci + 1);
        int qx, qy, tag = lane, dummy = 0;
        bool valid;
        if (lane == 0)      { qx = pmvx; qy = pmvy; valid = true; }
        else if (lane == 1) { qx = bmx * 4; qy = bmy * 4; valid = ((pmvx & 3) | (pmvy & 3)) != 0; }
        else if (lane == 2) { qx = 0; qy = 0; valid = (pmvx | pmvy) != 0; }
        else
        {
            qx = max(min(candx, qmaxx), qminx); qy = max(min(candy, qmaxy), qminy);
            valid = lane - 3 < j.numCand && (qx | qy) && !(qx == pmvx && qy == pmvy);
        }
        const int cnt = 3 + j.numCand;
        valid = valid && lane < cnt;
        const int n = me_compact(valid, cnt, qx, qy, tag, dummy);
        int cost = PL ? me_sad_points(c, n, me_qpel_off(c, qx, qy)) : me_subpel_batch<P, CLS>(c, n, qx, qy, false);
        if (CHROMA && cc->on)
        {
            // the clipped MVP and the candidates go through subpelCompare (chroma term included); the MVP's full-pel
            // rounding and MV 0 are plain COST_MV SADs (motion.cpp:771-814)
            const bool wantC = lane < n && (tag == 0 || tag >= 3);
            const int ccost = me_chroma_batch<P, CLS>(c, *cc, n, qx, qy, __ballot_sync(0xffffffffu, wantC));
            if (wantC) cost += ccost;
        }
        const bool mine = lane < n;
        const unsigned m0 = __ballot_sync(0xffffffffu, mine && tag == 0);
        const unsigned m1 = __ballot_sync(0xffffffffu, mine && tag == 1);
        const unsigned m2 = __ballot_sync(0xffffffffu, mine && tag == 2);
        bprecost = __shfl_sync(0xffffffffu, cost, __ffs(m0) - 1);
        bcost = bprecost;
        const int mvc1 = me_mvcost(c, bmx * 4, bmy * 4), mvc0 = me_mvcost(c, 0, 0);
        if (m1) bcost = __shfl_sync(0xffffffffu, cost, __ffs(m1) - 1) + mvc1;
        if (m2)
        {
            const int cz = __shfl_sync(0xffffffffu, cost, __ffs(m2) - 1) + mvc0;
            if (cz < bcost) { bcost = cz; bmx = 0; bmy = max(min(0, c.maxy), c.miny); }
        }
        const bool isCand = mine && tag >= 3;
        if (isCand) cost += me_mvcost(c, qx, qy);
        const unsigned key = isCand ? (((unsigned)cost << 5) | (unsigned)lane) : 0xffffffffu;
        const unsigned mk = __reduce_min_sync(0xffffffffu, key);
        if (mk != 0xffffffffu && (int)(mk >> 5) < bprecost)
        {
            bprecost = (int)(mk >> 5);
            bestprex = __shfl_sync(0xffffffffu, qx, (int)(mk & 31)); bestprey = __shfl_sync(0xffffffffu, qy, (int)(mk & 31));
        }
    }

    st.bmx = bmx; st.bmy = bmy; st.bcost = bcost; st.bprecost = bprecost; st.bestprex = bestprex; st.bestprey = bestprey;
}

// raster refinement (motion.cpp:1171-1201): grid of step 5 over the whole window.  Every 4th column of a row (when it
// closes a full x4 group) adds mvcost(tmv << 3) as in the reference.  Global-memory version: 32 points per burst.
template <typename P>
__device__ __forceinline__ void me_raster(const MeCtx<P>& c, MeStar& s)
{
    const int RD = 5;
    const int ncols = (c.maxx - c.minx) / RD + 1, nrows = (c.maxy - c.miny) / RD + 1;
    const int total = ncols * nrows;
    for (int base = 0; base < total; base += 32)
    {
        const int idx = min(base + c.lane, total - 1);
        const int rj = idx / ncols, ri = idx - rj * ncols;
        int px = c.minx + ri * RD, py = c.miny + rj * RD;
        const int n = min(32, total - base);
        const bool x8 = (ri & 3) == 3;
        int cost = me_eval_points(c, n, px, py, x8);
        const unsigned key = (unsigned)me_argmin(n, cost, c.lane);
        if ((int)(key >> 5) < s.bcost)
        {
            s.bcost = (int)(key >> 5);
            s.bx = __shfl_sync(0xffffffffu, px, (int)(key & 31)); s.by = __shfl_sync(0xffffffffu, py, (int)(key & 31));
        }
    }
}

// STAR (motion.cpp:1132-1240), written as one loop so that the star pattern, the two-point refinement and the raster scan
// each have exactly one (inlined) evaluation site.  Generic over the context: MeCtx (global-memory gathers) or MeWin
// (shared-memory search window, me_window.cuh); me_eval_points / me_raster are the per-context evaluation sites.
template <typename CTX>
__device__ __forceinline__ void me_star_search(const CTX& c, MeStar& s, int merange)
{
    bool first = true;
    for (;;)
    {
        me_star_pattern(c, s, first ? 3 : 32, merange, first);
        const bool d1 = s.dist == 1;
        bool improved = false;
        if (d1 && s.point)
        {
            // the two neighbours of the winning distance-1 point (motion.cpp:1139-1166 / :1215-1236), in order, strict '<'
            const int saved = s.bcost;
            const int o = (s.point - 1) * 2 + (c.lane & 1);
            int px = s.bx + c_star_off[o][0], py = s.by + c_star_off[o][1], pt = s.point, ds = s.dist;
            const bool valid = c.lane < 2 && ME_INRANGE(px, py);
            const int n = me_compact(valid, 2, px, py, pt, ds);
            if (n > 0)
            {
                const int cost = me_eval_points(c, n, px, py, false);
                me_fold(s, n, cost, px, py, pt, ds);
            }
            improved = s.bcost != saved;
        }
        if (first)
        {
            if (d1 && !improved) break;
            if (s.dist > 5) me_raster(c, s);
            first = false;
        }
        else if (d1) break;
        if (s.dist <= 0) break;
        s.dist = 0; s.point = 0;
    }
}

// phase 2 (motion.cpp:816-1438): the integer search proper
template <typename P>
__device__ __forceinline__ void me_phase2(MeCtx<P>& c, const x265cu_me_job& j, MeState& st)
{
    const int merange = j.merange;
    int bmx = st.bmx, bmy = st.bmy, bcost = st.bcost;
    if (j.method == 0)
    {   // DIA (motion.cpp:822-846): the four neighbours of every step are one burst; the reference's packed compare
        // ((cost << 4) + tag, smallest wins) is the burst's key
        bcost <<= 4;
        int i = merange;
        do
        {
            const int k = c.lane & 3;
            const int px = bmx + (k == 2 ? -1 : k == 3 ? 1 : 0), py = bmy + (k == 0 ? -1 : k == 1 ? 1 : 0);
            const int tag = k == 0 ? 1 : k == 1 ? 3 : k == 2 ? 4 : 12;
            const int cost = me_eval_points(c, 4, px, py, false);
            const bool ok = c.lane < 4 && (k >= 2 || ME_YOK(py));
            const unsigned key = ok ? (unsigned)((cost << 4) + tag) : 0xffffffffu;
            const unsigned m = __reduce_min_sync(0xffffffffu, key);
            if (m < (unsigned)bcost) bcost = (int)m;
            if (!(bcost & 15)) break;
            bmx -= (int)((unsigned)bcost << 28) >> 30;
            bmy -= (int)((unsigned)bcost << 30) >> 30;
            bcost &= ~15;
        }
        while (--i && ME_INRANGE(bmx, bmy));
        bcost >>= 4;
    }
    else if (j.method == 1)
    {   // HEX (motion.cpp:848-945), burst per step: the 6 hexagon points, then 3 new points per move, then the
        // 8-point square; keys are the reference's (cost << 3) + tag, ties to the smaller tag as in its compare chain
        const int lane = c.lane;
        {
            // tags 2..7 = hex2[1..6]: (-2,0) (-1,2) (1,2) (2,0) (1,-2) (-1,-2)
            const int k = min(lane, 5);
            const int px = bmx + c_hex2[k + 1][0], py = bmy + c_hex2[k + 1][1];
            const int cost = me_eval_points(c, 6, px, py, false);
            bcost <<= 3;
            const unsigned key = (lane < 6 && ME_YOK(py)) ? (unsigned)((cost << 3) + k + 2) : 0xffffffffu;
            const unsigned m = __reduce_min_sync(0xffffffffu, key);
            if (m < (unsigned)bcost) bcost = (int)m;
        }
        if (bcost & 7)
        {
            int dir = (bcost & 7) - 2;
            if (ME_YOK(bmy + c_hex2[dir + 1][1]))
            {
                bmx += c_hex2[dir + 1][0]; bmy += c_hex2[dir + 1][1];
                for (int i = (merange >> 1) - 1; i > 0 && ME_INRANGE(bmx, bmy); i--)
                {
                    const int k = min(lane, 2);
                    const int px = bmx + c_hex2[dir + k][0], py = bmy + c_hex2[dir + k][1];
                    const int cost = me_eval_points(c, 3, px, py, false);
                    bcost &= ~7;
                    const unsigned key = (lane < 3 && ME_YOK(py)) ? (unsigned)((cost << 3) + k + 1) : 0xffffffffu;
                    const unsigned m = __reduce_min_sync(0xffffffffu, key);
                    if (m < (unsigned)bcost) bcost = (int)m;
                    if (!(bcost & 7)) break;
                    dir += (bcost & 7) - 2;
                    dir = c_mod6m1[dir + 1];
                    bmx += c_hex2[dir + 1][0]; bmy += c_hex2[dir + 1][1];
                }
            }
        }
        bcost >>= 3;
        {
            // square refine: square1[1..8] in order, strict '<' (x is not range-checked by the reference, y is)
            const int k = min(lane, 7) + 1;
            const int px = bmx + c_square1[k][0], py = bmy + c_square1[k][1];
            const int cost = me_eval_points(c, 8, px, py, false);
            const bool ok = lane < 8 && (c_square1[k][1] == 0 || ME_YOK(py));
            const unsigned key = ok ? (((unsigned)cost << 5) | (unsigned)lane) : 0xffffffffu;
            const unsigned m = __reduce_min_sync(0xffffffffu, key);
            int dir = 0;
            if (m != 0xffffffffu && (int)(m >> 5) < bcost) { bcost = (int)(m >> 5); dir = (int)(m & 31) + 1; }
            bmx += c_square1[dir][0]; bmy += c_square1[dir][1];
        }
    }
    else if (j.method == 5)
    {   // X265_FULL_SEARCH (motion.cpp:1397-1440): every full-pel position of [mvmin, mvmax] in raster order with a strict '<':
        // bursts of 32 consecutive x positions; a burst's winner is its minimum with ties to the lowest x, which is the
        // position the sequential compare would keep, and it replaces the best so far only when strictly cheaper
        for (int ty = c.miny; ty <= c.maxy; ty++)
            for (int tx0 = c.minx; tx0 <= c.maxx; tx0 += 32)
            {
                const int n = min(32, c.maxx - tx0 + 1);
                const int px = tx0 + min(c.lane, n - 1);
                const int cost = me_eval_points(c, n, px, ty, false);
                const unsigned key = c.lane < n ? (((unsigned)cost << 5) | (unsigned)c.lane) : 0xffffffffu;
                const unsigned m = __reduce_min_sync(0xffffffffu, key);
                if ((int)(m >> 5) < bcost) { bcost = (int)(m >> 5); bmx = tx0 + (int)(m & 31); bmy = ty; }
            }
    }
    else
    {
        MeStar s; s.bx = bmx; s.by = bmy; s.bcost = bcost; s.point = 0; s.dist = 0;
        me_star_search(c, s, merange);
        bmx = s.bx; bmy = s.by; bcost = s.bcost;
    }

    st.bmx = bmx; st.bmy = bmy; st.bcost = bcost;
}

// phase 3 (motion.cpp:1440-1569): pick pre-check vs search winner, sub-pel refinement (PL: out of the phase planes)
template <typename P, int CLS, bool CHROMA = false, bool PL = false>
__device__ __forceinline__ void me_phase3(MeCtx<P>& c, const x265cu_me_job& j, const MeState& st, int32_t* __restrict__ out, const MeChromaCtx<P>* cc = nullptr)
{
    const int qminy = c.miny * 4, qmaxy = c.maxy * 4;
    int bcost = st.bcost;
    const int bmx = st.bmx, bmy = st.bmy, bprecost = st.bprecost, bestprex = st.bestprex, bestprey = st.bestprey;
    int bx, by;
    if (bprecost < bcost) { bx = bestprex; by = bestprey; bcost = bprecost; }
    else { bx = bmx * 4; by = bmy * 4; }
    const int8_t* wl = c_workload[j.subme];
    if (!bcost)
        bcost = me_mvcost(c, bx, by);
    else if (c.lowres)
    {
        // half-pel round (SAD), SATD at the winner, quarter-pel round (SATD): each round is one burst over the lowres planes
        for (int rnd = 0; rnd < 2; rnd++)
        {
            const int dirs = rnd ? wl[3] : wl[1], step = rnd ? 1 : 2;
            if (rnd)
            {
                const int cc = me_lowres_multi(c, 1, bx, by, true);
                bcost = __shfl_sync(0xffffffffu, cc, 0) + me_mvcost(c, bx, by);
            }
            const int i1 = min(c.lane + 1, 8);
            int qx = bx + c_square1[i1][0] * step, qy = by + c_square1[i1][1] * step, dir = i1, dummy = 0;
            const bool valid = c.lane < dirs && !((qy < qminy) | (qy > qmaxy));
            const int n = me_compact(valid, dirs, qx, qy, dir, dummy);
            int cost = me_lowres_batch(c, n, qx, qy, rnd != 0);
            if (c.lane < n) cost += me_mvcost(c, qx, qy);
            int bdir = 0;
            if (n > 0)
            {
                const unsigned key = (unsigned)me_argmin(n, cost, c.lane);
                if ((int)(key >> 5) < bcost) { bcost = (int)(key >> 5); bdir = __shfl_sync(0xffffffffu, dir, (int)(key & 31)); }
            }
            bx += c_square1[bdir][0] * step; by += c_square1[bdir][1] * step;
        }
    }
    else
    {
        // motion.cpp:1496-1558 as one loop with a single (inlined) evaluation site: stage 0 = SATD at the start point
        // (when the half-pel rounds use SATD), stage 1 = half-pel rounds, stage 2 = SATD at the half-pel winner
        // (otherwise), stage 3 = quarter-pel rounds.  A "centre" step is a burst of one candidate.
        const bool hsatd = wl[4] != 0;
        int stage = hsatd ? 0 : 1, it = 0;
        for (;;)
        {
            if (stage == 1 && it >= wl[0]) { stage = hsatd ? 3 : 2; it = 0; }
            if (stage == 3 && it >= wl[2]) break;
            const bool centre = (stage & 1) == 0;
            const int dirs = centre ? 1 : (stage == 1 ? wl[1] : wl[3]), step = stage == 1 ? 2 : 1;
            const bool satd = stage == 1 ? hsatd : true;
            const int i1 = centre ? 0 : min(c.lane + 1, 8);
            int qx = bx + c_square1[i1][0] * step, qy = by + c_square1[i1][1] * step, dir = i1, dummy = 0;
            const bool valid = c.lane < dirs && (centre || !((qy < qminy) | (qy > qmaxy)));
            const int n = me_compact(valid, dirs, qx, qy, dir, dummy);
            int cost = me_subpel_batch<P, CLS, PL>(c, n, qx, qy, satd);
            if (CHROMA && cc->on)
            {
                const int ccost = me_chroma_batch<P, CLS>(c, *cc, n, qx, qy, n >= 32 ? 0xffffffffu : ((1u << n) - 1u));
                if (c.lane < n) cost += ccost;
            }
            if (c.lane < n) cost += me_mvcost(c, qx, qy);
            if (centre) { bcost = __shfl_sync(0xffffffffu, cost, 0); stage++; continue; }
            int bdir = 0;
            if (n > 0)
            {
                const unsigned key = (unsigned)me_argmin(n, cost, c.lane);
                if ((int)(key >> 5) < bcost) { bcost = (int)(key >> 5); bdir = __shfl_sync(0xffffffffu, dir, (int)(key & 31)); }
            }
            if (bdir) { bx += c_square1[bdir][0] * step; by += c_square1[bdir][1] * step; it++; }
            else if (stage == 1) { stage = hsatd ? 3 : 2; it = 0; }
            else break;
        }
    }
    if (c.lane == 0) { out[0] = bcost; out[1] = bx; out[2] = by; out[3] = 0; }
}


template <typename P>
__device__ __forceinline__ void me_run_job(MeCtx<P>& c, const x265cu_me_job& j, int32_t* __restrict__ out)
{
    MeState st;
    me_phase1<P, -1>(c, j, st);
    me_phase2<P>(c, j, st);
    me_phase3<P, -1>(c, j, st, out);
}

// Job setup shared by all ME kernels
template <typename P>
__device__ __forceinline__ void me_make_ctx(MeCtx<P>& c, const x265cu_me_job& j, const P* fenc, int fstride, const P* const* refs, int rstride,
                                            int lowres, const uint16_t* mvcost, int lane, MeShared* sm)
{
    c.fenc = fenc + j.offset; c.fstride = fstride;
    if (lowres) { for (int i = 0; i < 4; i++) c.ref[i] = refs[j.ref * 4 + i] + j.offset; }
    else        { c.ref[0] = refs[j.ref] + j.offset; c.ref[1] = c.ref[2] = c.ref[3] = c.ref[0]; }
    c.rstride = rstride; c.mvc = mvcost;
    c.mvpx = j.qmvp[0]; c.mvpy = j.qmvp[1];
    c.minx = j.mvmin[0]; c.miny = j.mvmin[1]; c.maxx = j.mvmax[0]; c.maxy = j.mvmax[1];
    c.w = j.pw; c.h = j.ph; c.lgw = 31 - __clz(c.w); c.lane = lane; c.lowres = lowres; c.sm = sm; c.ppitch = 0;
    c.pow2 = ((c.w & (c.w - 1)) | (c.h & (c.h - 1))) == 0;
    const int wpr = (c.w * (int)sizeof(P)) >> 2;            // words per row (>= 1: w >= 4)
    c.lgwpr = 31 - __clz(wpr);
    c.nw = wpr * c.h; c.lgnw = 31 - __clz(c.nw);
    // widest lane segment (16 / 8 / 4 bytes) that both a PU row and the fenc row alignment allow
    const unsigned fal = (unsigned)(uintptr_t)c.fenc | (unsigned)(fstride * (int)sizeof(P));
    c.lgsegw = min(c.lgwpr, (fal & 15u) == 0 ? 2 : (fal & 7u) == 0 ? 1 : 0);
    if ((unsigned)(rstride * (int)sizeof(P)) & 7u) c.lgsegw = 0;        // the 8-byte aligned reference loads need an 8-byte row pitch
}

// Persistent warps with a dynamic job queue (jobs differ by up to 64x in work).  The search is split into
// launches -- pre-checks (small PUs, other PUs), integer search, sub-pel refinement (small PUs, other PUs) --
// because the fused body (12.4 K SASS instructions, ~200 KB) thrashes the instruction cache: ncu
// showed 80 % of the stall samples in `no_instructions` at a 46 % i-cache hit rate, and the un-split sub-pel
// kernel (8.8 K instructions, both PU classes resident on every SM) still sat at 64 %.  PHASE 0 = all fused
// (the lookahead kernel's per-CU call).  PL (pre-check and sub-pel launches of the frame analyser): candidates are read
// from the quarter-pel phase planes `ppitch` bytes apart in every reference allocation; no shared-memory scratch.
#ifndef ME_MIN_BLOCKS
#define ME_MIN_BLOCKS 3
#endif
#ifndef ME_P2_BLOCKS
#define ME_P2_BLOCKS 4
#endif
#ifndef ME_BIG_BLOCKS
#define ME_BIG_BLOCKS 2          // large-PU pre-check / sub-pel kernels: 128 registers beat a third resident CTA (no spills in the tap loops)
#endif
template <typename P, int PHASE, int CLS, bool PL = false>
__global__ void __launch_bounds__(256, PHASE == 2 ? ME_P2_BLOCKS : (CLS == 1 ? ME_BIG_BLOCKS : ME_MIN_BLOCKS)) k_me(const P* __restrict__ fenc, int fstride, const P* const* __restrict__ refs, int rstride, int lowres,
                                                           const uint16_t* __restrict__ mvcost, const x265cu_me_job* __restrict__ jobs, int n,
                                                           int32_t* __restrict__ out, MeState* __restrict__ state, int* __restrict__ counter,
                                                           const int32_t* __restrict__ list = nullptr, const int* __restrict__ list_n = nullptr,
                                                           const int32_t* __restrict__ order = nullptr, int order0 = 0, int ppitch = 0)
{
    extern __shared__ unsigned char me_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    MeShared* sm = (MeShared*)me_smem + warp;
    // with `list`: the jobs are list[0 .. *list_n) (the leftovers of the shared-memory-window search, me_window.cuh)
    if (list) n = *list_n;
    for (;;)
    {
        int jid = 0;
        if (lane == 0) jid = atomicAdd(counter, 1);
        jid = __shfl_sync(0xffffffffu, jid, 0);
        if (jid >= n) break;
        if (list) jid = list[jid];
        // `order`: the launch slice's jobs sorted by PU shape (absolute job indices, slice start order0): the warps of the whole
        // GPU then run the same PU size -- the same code paths -- at the same time (the kernels are instruction-cache bound)
        if (order) jid = order[jid] - order0;
        const x265cu_me_job j = jobs[jid];
        MeCtx<P> c;
        me_make_ctx<P>(c, j, fenc, fstride, refs, rstride, lowres, mvcost, lane, sm);
        if (PL) c.ppitch = ppitch;
        if (CLS >= 0 && me_subpel_class(c) != CLS) continue;                   // the sibling launch owns this job
        if (PHASE == 0) me_run_job<P>(c, j, out + (size_t)jid * 4);
        else
        {
            MeState st;
            if (PHASE != 1) st = state[jid];
            if (PHASE == 1) { me_phase1<P, CLS, false, PL>(c, j, st); if (lane == 0) state[jid] = st; }
            if (PHASE == 2) { me_phase2<P>(c, j, st); if (lane == 0) state[jid] = st; }
            if (PHASE == 3) me_phase3<P, CLS, false, PL>(c, j, st, out + (size_t)jid * 4);
        }
        __syncwarp();
    }
}

// The pre-check and sub-pel launches with the chroma-SATD term (x265cu_me_batch_chroma): separate instantiations, so
// the luma-only kernels above are unchanged by it.  The integer search (phase 2) is luma only in the reference too.
template <typename P, int PHASE, int CLS, bool PL = false>
__global__ void __launch_bounds__(256, CLS == 1 ? ME_BIG_BLOCKS : ME_MIN_BLOCKS) k_me_chroma(const P* __restrict__ fenc, int fstride, const P* const* __restrict__ refs, int rstride,
                                                           MeChromaArgs ch, const uint16_t* __restrict__ mvcost, const x265cu_me_job* __restrict__ jobs, int n,
                                                           int32_t* __restrict__ out, MeState* __restrict__ state, int* __restrict__ counter,
                                                           const int32_t* __restrict__ order = nullptr, int order0 = 0, int ppitch = 0)
{
    extern __shared__ unsigned char me_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    MeShared* sm = (MeShared*)me_smem + warp;
    for (;;)
    {
        int jid = 0;
        if (lane == 0) jid = atomicAdd(counter, 1);
        jid = __shfl_sync(0xffffffffu, jid, 0);
        if (jid >= n) break;
        if (order) jid = order[jid] - order0;          // shape-sorted job order (see k_me)
        const x265cu_me_job j = jobs[jid];
        MeCtx<P> c;
        me_make_ctx<P>(c, j, fenc, fstride, refs, rstride, 0, mvcost, lane, sm);
        if (PL) c.ppitch = ppitch;
        if (me_subpel_class(c) != CLS) continue;                   // the sibling launch owns this job
        MeChromaCtx<P> cc;
        me_set_chroma<P>(cc, c, j, ch, fstride);
        MeState st;
        if (PHASE == 1) { me_phase1<P, CLS, true, PL>(c, j, st, &cc); if (lane == 0) state[jid] = st; }
        else            { st = state[jid]; me_phase3<P, CLS, true, PL>(c, j, st, out + (size_t)jid * 4, &cc); }
        __syncwarp();
    }
}

template <typename P, int PHASE, int CLS, bool PL = false>
static int launch_me_chroma_phase(x265cu_ctx* ctx, const void* fenc, int fstride, const void* const* refs, int rstride, const MeChromaArgs& ch,
                                  const uint16_t* mvcost, const x265cu_me_job* jobs, int n, int32_t* out, MeState* state, int* counter,
                                  const int32_t* order = NULL, int order0 = 0, int ppitch = 0)
{
    const int threads = 256, warps = threads / 32;
    const size_t smem = PL ? 0 : sizeof(MeShared) * warps;            // the phase-plane path never touches the interpolation scratch
    int blocks = ctx->sm_count * (CLS == 1 ? ME_BIG_BLOCKS : ME_MIN_BLOCKS);
    int need = (n + warps - 1) / warps;
    if (blocks > need) blocks = need;
    k_me_chroma<P, PHASE, CLS, PL><<<blocks, threads, smem, ctx->stream>>>((const P*)fenc, fstride, (const P* const*)refs, rstride, ch, mvcost, jobs, n, out, state, counter, order, order0, ppitch);
    CU_LAUNCH_CHECK(ctx);
    return 0;
}

template <typename P, int PHASE, int CLS, bool PL = false>
static int launch_me_phase(x265cu_ctx* ctx, const void* fenc, int fstride, const void* const* refs, int rstride, int lowres,
                           const uint16_t* mvcost, const x265cu_me_job* jobs, int n, int32_t* out, MeState* state, int* counter,
                           const int32_t* list = NULL, const int* list_n = NULL, const int32_t* order = NULL, int order0 = 0, int ppitch = 0)
{
    const int threads = 256, warps = threads / 32;
    // the integer search and the phase-plane path never touch the interpolation scratch
    const size_t smem = (PHASE == 2 || PL) ? 0 : sizeof(MeShared) * warps;
    int blocks = ctx->sm_count * (PHASE == 2 ? ME_P2_BLOCKS : (CLS == 1 ? ME_BIG_BLOCKS : ME_MIN_BLOCKS));
    int need = (n + warps - 1) / warps;
    if (blocks > need) blocks = need;
    k_me<P, PHASE, CLS, PL><<<blocks, threads, smem, ctx->stream>>>((const P*)fenc, fstride, (const P* const*)refs, rstride, lowres, mvcost, jobs, n, out, state, counter, list, list_n, order, order0, ppitch);
    CU_LAUNCH_CHECK(ctx);
    return 0;
}

// Shared-memory-window integer search (me_window.cuh): the caller (the frame analyser) owns the group tables and the tensor
// maps of its reference planes; `left_*` receive the jobs the window kernel hands back to the global-memory kernel.
struct MeWinLaunch
{
    const void* tmaps; int allocX, allocY;                  // device array [ref][MEW_NCLS] of CUtensorMap; picture origin inside the allocation
    const void* groups[3]; int ngroups[3];                  // MeGroup lists of the launch slice: [0] CU 64 groups, [1] CU 32 groups, [2] 16x16 cells
    const int32_t* grp_jobs[3]; int job0;                   // absolute job indices; job0 = first job of the slice
    int amp;                                                // AMP partitions present (13 PUs per CU instead of 5): sizes the CTAs
    const int32_t* order;                                   // the slice's jobs sorted by PU shape (absolute indices) or NULL
    int* left_count; int32_t* left_list;
};
template <typename P>
static int launch_me_window(x265cu_ctx* ctx, const void* fenc, int fstride, const uint16_t* mvcost, const x265cu_me_job* jobs,
                            MeState* st, const MeWinLaunch& w);

// the two PU-class launches (small pow2 PUs, everything else) of a pre-check (PHASE 1) or sub-pel (PHASE 3) pass;
// `counter_dev` = the first of their two job counters
template <typename P, int PHASE, bool PL>
static int launch_me_classes(x265cu_ctx* ctx, const void* fenc, int fstride, const void* const* refs, int rstride, int lowres,
                             const uint16_t* mvcost, const x265cu_me_job* jobs, int n, int32_t* out, MeState* st, int* counter_dev,
                             const MeChromaArgs* ch, const int32_t* ord, int ord0, int ppitch)
{
    int rc = 0;
    if (ch)
    {
        rc |= launch_me_chroma_phase<P, PHASE, 0, PL>(ctx, fenc, fstride, refs, rstride, *ch, mvcost, jobs, n, out, st, counter_dev + 0, ord, ord0, ppitch);
        rc |= launch_me_chroma_phase<P, PHASE, 1, PL>(ctx, fenc, fstride, refs, rstride, *ch, mvcost, jobs, n, out, st, counter_dev + 1, ord, ord0, ppitch);
    }
    else
    {
        rc |= launch_me_phase<P, PHASE, 0, PL>(ctx, fenc, fstride, refs, rstride, lowres, mvcost, jobs, n, out, st, counter_dev + 0, NULL, NULL, ord, ord0, ppitch);
        rc |= launch_me_phase<P, PHASE, 1, PL>(ctx, fenc, fstride, refs, rstride, lowres, mvcost, jobs, n, out, st, counter_dev + 1, NULL, NULL, ord, ord0, ppitch);
    }
    return rc;
}

// ppitch != 0: the references carry quarter-pel phase planes ppitch bytes apart (frame analyser); the pre-check and
// sub-pel launches then read their candidates from them
template <typename P>
static int launch_me_t(x265cu_ctx* ctx, const void* fenc, int fstride, const void* const* refs, int rstride, int lowres,
                       const uint16_t* mvcost, const x265cu_me_job* jobs, int n, int32_t* out, MeState* st, int* counter_dev,
                       const MeChromaArgs* ch, const MeWinLaunch* win, int ppitch)
{
    int rc = 0;
    // shape-sorted job order (geometry.h `order`), measured on B200 at 2160p (profiles/me_r2_ncu.md section 5): it helps kernels
    // that miss the instruction cache (the chroma sub-pel launches: 24.2 -> 23.2 ms; 36.7 -> 27.6 ms before the column-split
    // chroma term made them small) and costs the others ~10 % (they lose the raster order's L1 / L2 locality: luma-only
    // pre-checks 9.1 -> 10.4 ms, chroma pre-checks 9.7 -> 10.9 ms).  X265CU_ME_ORDER = 0: never, 1: chroma sub-pel launches
    // only (default), 2: every pre-check / sub-pel launch.
    static const int ordMode = [] { const char* e = getenv("X265CU_ME_ORDER"); return e ? atoi(e) : 1; }();
    const int32_t* ordAll = (win && !lowres) ? win->order : NULL;
    const int32_t* ord = ordMode >= 2 ? ordAll : NULL;                       // pre-checks, luma-only sub-pel
    const int32_t* ord3 = (ordMode >= 2 || (ordMode == 1 && ch)) ? ordAll : NULL;   // chroma sub-pel
    const int ord0 = win ? win->job0 : 0;
    rc |= ppitch ? launch_me_classes<P, 1, true>(ctx, fenc, fstride, refs, rstride, lowres, mvcost, jobs, n, out, st, counter_dev + 0, ch, ord, ord0, ppitch)
                 : launch_me_classes<P, 1, false>(ctx, fenc, fstride, refs, rstride, lowres, mvcost, jobs, n, out, st, counter_dev + 0, ch, ord, ord0, 0);
    CU_CHECK(cudaEventRecord(ctx->me_ev[1], ctx->stream));
    if (win && !lowres)
    {
        // STAR groups out of shared-memory windows; whatever does not fit (or is not STAR) through the global-memory kernel
        rc |= launch_me_window<P>(ctx, fenc, fstride, mvcost, jobs, st, *win);
        rc |= launch_me_phase<P, 2, -1>(ctx, fenc, fstride, refs, rstride, lowres, mvcost, jobs, n, out, st, counter_dev + 2, win->left_list, win->left_count);
    }
    else
        rc |= launch_me_phase<P, 2, -1>(ctx, fenc, fstride, refs, rstride, lowres, mvcost, jobs, n, out, st, counter_dev + 2);
    CU_CHECK(cudaEventRecord(ctx->me_ev[2], ctx->stream));
    const int32_t* ordS = ch ? ord3 : ord;
    rc |= ppitch ? launch_me_classes<P, 3, true>(ctx, fenc, fstride, refs, rstride, lowres, mvcost, jobs, n, out, st, counter_dev + 3, ch, ordS, ord0, ppitch)
                 : launch_me_classes<P, 3, false>(ctx, fenc, fstride, refs, rstride, lowres, mvcost, jobs, n, out, st, counter_dev + 3, ch, ordS, ord0, 0);
    return rc;
}

static int launch_me(x265cu_ctx* ctx, int depth, const void* fenc, int fstride, const void* const* refs, int rstride, int lowres,
                     const uint16_t* mvcost, const x265cu_me_job* jobs, int n, int32_t* out, int* counter_dev, const MeChromaArgs* chroma = NULL,
                     const MeWinLaunch* win = NULL, int ppitch = 0)
{
    if (n <= 0) return 0;
    CU_CHECK(cudaMemsetAsync(counter_dev, 0, 8 * sizeof(int), ctx->stream));
    // per-job state between the phases (24 B per job), grown on demand and kept by the context
    const size_t need = (size_t)n * sizeof(MeState);
    if (ctx->me_state_bytes < need)
    {
        if (ctx->d_me_state) { CU_CHECK(cudaStreamSynchronize(ctx->stream)); cudaFree(ctx->d_me_state); }
        CU_CHECK(cudaMalloc(&ctx->d_me_state, need));
        ctx->me_state_bytes = need;
    }
    MeState* st = (MeState*)ctx->d_me_state;
    CU_CHECK(cudaEventRecord(ctx->me_ev[0], ctx->stream));
    if (chroma && lowres) chroma = NULL;                    // the lowres planes have no chroma (lowres.h)
    if (lowres) ppitch = 0;
    const int rc = depth == 8 ? launch_me_t<uint8_t>(ctx, fenc, fstride, refs, rstride, lowres, mvcost, jobs, n, out, st, counter_dev, chroma, win, ppitch)
                              : launch_me_t<uint16_t>(ctx, fenc, fstride, refs, rstride, lowres, mvcost, jobs, n, out, st, counter_dev, chroma, win, ppitch);
    CU_CHECK(cudaEventRecord(ctx->me_ev[3], ctx->stream));
    return rc;
}
