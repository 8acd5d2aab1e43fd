// x265_b200/csrc/phase_planes.cuh -- quarter-pel phase planes of the frame analyser's references.
// HEVC luma interpolation of a block depends only on the pixel position and the fractional phase (ipfilter.cpp:
// luma_hpp, luma_vpp, luma_hvpp = hps(rowExt) + vsp), so the 15 fractional phases of a reference can be computed once
// per pixel and every sub-pel candidate of the motion search becomes a full-pel compare on one of them (me.cuh, PL).
// Plane (yFrac << 2) | xFrac of reference r lives `ppitch` bytes after plane 0 (the reference itself) in the same
// allocation, with the same stride and margins.
#pragma once
#include "common.cuh"
#include "interp.cuh"
#include "phase_planes.h"
#include <limits.h>

// Union of the job boxes (phase_planes.h) per reference: box[4 * ref + {0, 1, 2, 3}] = {x0, -x1, y0, -y1}, all minima,
// so one atomicMin per entry; the caller initialises them to INT_MAX.  Per-CTA reduction in shared memory first.
__global__ void __launch_bounds__(256) k_phase_plane_box(const x265cu_me_job* __restrict__ jobs, int n, int stride, int* __restrict__ box)
{
    __shared__ int sbox[16 * 4];
    for (int k = threadIdx.x; k < 16 * 4; k += blockDim.x) sbox[k] = INT_MAX;
    __syncthreads();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n)
    {
        const x265cu_me_job j = jobs[i];
        const int y = j.offset / stride, x = j.offset - y * stride;
        int b[4];
        phase_plane_job_box(x, y, j.pw, j.ph, j.mvmin[0], j.mvmin[1], j.mvmax[0], j.mvmax[1], b);
        int* s = sbox + 4 * j.ref;
        atomicMin(s + 0, b[0]); atomicMin(s + 1, -b[1]); atomicMin(s + 2, b[2]); atomicMin(s + 3, -b[3]);
    }
    __syncthreads();
    for (int k = threadIdx.x; k < 16 * 4; k += blockDim.x)
        if (sbox[k] != INT_MAX) atomicMin(box + k, sbox[k]);
}

#define PP_TW 64                            // output tile: 64 columns (16 lanes x 4 pixels) x 16 rows, 256 threads
#define PP_TH 16

// Writes planes 1..15 of every reference (grid.z = reference) over the reference's box, clipped to the region of
// phase_plane_region() (x < regX1, y < regY1).  Grid x / y tile that region from its top-left corner (-PP_PAD, -PP_PAD).
// `ref0[r]` = pixel (0, 0) of reference r's plane 0; (lastX, lastY) = the last pixel inside the allocation.
// A CTA stages its tile's source pixels plus the 8-tap support (3 before, 4 after) and the three horizontal phases of
// every staged row as the int16 rowExt intermediate (hps, kind 1); each lane then emits 4 adjacent pixels of one row in all 15 phases: 3 h (hpp), 3 v (vpp) and 9 hv (vsp over the intermediate),
// with the rounding of interp_finish, i.e. the bytes subpelCompare builds (motion.cpp:1571-1598).
template <typename P>
__global__ void __launch_bounds__(256) k_luma_phase_planes(uint8_t* const* __restrict__ ref0, int stride, size_t ppitch,
                                                           const int* __restrict__ box, int regX1, int regY1, int lastX, int lastY)
{
    constexpr int DEPTH = PixTraits<P>::depth;
    constexpr int SW = PP_TW + 8, SH = PP_TH + 7;
    __shared__ int16_t src[SH][SW];
    __shared__ __align__(16) int16_t mid[3][SH][PP_TW];
    const int r = blockIdx.z;
    const int tx0 = -PP_PAD + (int)blockIdx.x * PP_TW, ty0 = -PP_PAD + (int)blockIdx.y * PP_TH;
    // the reference's box, clipped to the region; whole CTA out when the tile misses it
    const int bx0 = max(box[4 * r + 0], -PP_PAD), bx1 = min(-box[4 * r + 1], regX1);
    const int by0 = max(box[4 * r + 2], -PP_PAD), by1 = min(-box[4 * r + 3], regY1);
    if (tx0 >= bx1 || tx0 + PP_TW <= bx0 || ty0 >= by1 || ty0 + PP_TH <= by0) return;
    const P* base = (const P*)ref0[r];
    const int tid = threadIdx.x;
    // source pixels: rows ty0 - 3 .. ty0 + PP_TH + 3, columns tx0 - 3 .. tx0 + PP_TW + 3.  The margins are at least PP_PAD + 4
    // pixels, so every pixel that a stored output reads is inside the allocation; the clamp only keeps the last tiles'
    // unused rows / columns from reading past it.
    for (int i = tid; i < SH * (PP_TW + 7); i += 256)
    {
        const int sy = i / (PP_TW + 7), sx = i - sy * (PP_TW + 7);
        src[sy][sx] = (int16_t)__ldg(base + (ptrdiff_t)min(ty0 - 3 + sy, lastY) * stride + min(tx0 - 3 + sx, lastX));
    }
    __syncthreads();
    // horizontal phases of every staged row as the hps intermediate
    for (int i = tid; i < SH * PP_TW; i += 256)
    {
        const int sy = i / PP_TW, sx = i - sy * PP_TW;
        int s[8];
#pragma unroll
        for (int k = 0; k < 8; k++) s[k] = src[sy][sx + k];
#pragma unroll
        for (int xf = 1; xf < 4; xf++)
        {
            int sum = 0;
#pragma unroll
            for (int k = 0; k < 8; k++) sum += s[k] * c_lumaFilter[xf][k];
            mid[xf - 1][sy][sx] = (int16_t)interp_finish<DEPTH>(sum, 1);
        }
    }
    __syncthreads();
    const int oy = tid >> 4, ox = (tid & 15) * 4;                // my 4 pixels: tile row oy, columns ox .. ox + 3
    const int py = ty0 + oy, px = tx0 + ox;
    if (py < by0 || py >= by1 || px + 4 <= bx0 || px >= bx1) return;
    int out[16][4];
    // h: hpp from the staged row (kind 0)
    {
        int s[11];
#pragma unroll
        for (int k = 0; k < 11; k++) s[k] = src[oy + 3][ox + k];
#pragma unroll
        for (int xf = 1; xf < 4; xf++)
#pragma unroll
            for (int q = 0; q < 4; q++)
            {
                int sum = 0;
#pragma unroll
                for (int k = 0; k < 8; k++) sum += s[q + k] * c_lumaFilter[xf][k];
                out[xf][q] = interp_finish<DEPTH>(sum, 0);
            }
    }
    // v: vpp from the staged columns (kind 0)
#pragma unroll
    for (int q = 0; q < 4; q++)
    {
        int s[8];
#pragma unroll
        for (int k = 0; k < 8; k++) s[k] = src[oy + k][ox + q + 3];
#pragma unroll
        for (int yf = 1; yf < 4; yf++)
        {
            int sum = 0;
#pragma unroll
            for (int k = 0; k < 8; k++) sum += s[k] * c_lumaFilter[yf][k];
            out[yf << 2][q] = interp_finish<DEPTH>(sum, 0);
        }
    }
    // hv: vsp over the intermediate (kind 2)
#pragma unroll
    for (int xf = 1; xf < 4; xf++)
#pragma unroll
        for (int q = 0; q < 4; q++)
        {
            int m[8];
#pragma unroll
            for (int k = 0; k < 8; k++) m[k] = mid[xf - 1][oy + k][ox + q];
#pragma unroll
            for (int yf = 1; yf < 4; yf++)
            {
                int sum = 0;
#pragma unroll
                for (int k = 0; k < 8; k++) sum += m[k] * c_lumaFilter[yf][k];
                out[(yf << 2) | xf][q] = interp_finish<DEPTH>(sum, 2);
            }
        }
    // one 4-pixel store per plane (4 B for 8-bit, 8 B for 16-bit pixels; px is a multiple of 4 and the plane origin
    // and stride are 4-pixel aligned)
    uint8_t* dst = (uint8_t*)(base + (ptrdiff_t)py * stride + px);
#pragma unroll
    for (int ph = 1; ph < 16; ph++)
    {
        uint8_t* d = dst + (size_t)ph * ppitch;
        if (sizeof(P) == 1)
            *(uint32_t*)d = (uint32_t)out[ph][0] | ((uint32_t)out[ph][1] << 8) | ((uint32_t)out[ph][2] << 16) | ((uint32_t)out[ph][3] << 24);
        else
            *(uint2*)d = make_uint2((uint32_t)out[ph][0] | ((uint32_t)out[ph][1] << 16), (uint32_t)out[ph][2] | ((uint32_t)out[ph][3] << 16));
    }
}
