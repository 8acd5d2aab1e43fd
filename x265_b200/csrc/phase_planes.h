// x265_b200/csrc/phase_planes.h -- which positions of the quarter-pel phase planes a motion search can read.
// Plain C++ (host and device): the frame analyser sizes and bounds the plane build with it, tests/phase_planes_capi.cpp
// exposes the same arithmetic to the CPU tests.
#pragma once
#ifdef __CUDACC__
#define PP_HD __host__ __device__
#else
#define PP_HD
#endif

// every job box of a picture lies inside [-PP_PAD, width + PP_PAD) x [-PP_PAD, height + PP_PAD) (phase_plane_region)
#define PP_PAD 76

static inline PP_HD int pp_min(int a, int b) { return a < b ? a : b; }
static inline PP_HD int pp_max(int a, int b) { return a > b ? a : b; }

// Rectangle box = {x0, x1, y0, y1} (half-open, picture pixels) of the phase-plane positions that the pre-checks and the
// sub-pel refinement of ONE job can read: the PU at picture pixel (x, y), w x h, full-pel search range [minx, maxx] x
// [miny, maxy] (x265cu_me_job.mvmin / mvmax).  A candidate (qx, qy) reads the w x h block at (qx >> 2, qy >> 2).
//   y: the pre-check candidates are clipped to the range, the sub-pel rounds drop candidates outside it, and MV 0 (always
//      pre-checked; its winner's y is clipped) is the only other start point: qy >> 2 in [min(miny, 0), max(maxy, 0)].
//   x: MV 0 again; the DIA / HEX steps move x without a range check (motion.cpp:822-945), at most 3 full-pels beyond it
//      (a hexagon move of 2, then the square refinement's 1), and the sub-pel rounds move x up to 6 quarter-pels (two
//      half-pel and two quarter-pel iterations, motion.cpp:48-58) unchecked: qx >> 2 in [min(minx, 0) - 5, max(maxx, 0) + 4].
static inline PP_HD void phase_plane_job_box(int x, int y, int w, int h, int minx, int miny, int maxx, int maxy, int box[4])
{
    box[0] = x + pp_min(minx, 0) - 5;
    box[1] = x + w + pp_max(maxx, 0) + 5;
    box[2] = y + pp_min(miny, 0);
    box[3] = y + h + pp_max(maxy, 0);
}

// The region every job box lies in: k_build_me_jobs clips the range to mvmin >= -(64 + 8 + cuX - 1) and
// mvmax <= width + 8 - cuX - 1 (cudata.cpp:1915-1928 clipMv), with the PU inside a CU of at most 64 pixels, so
// x0 >= -71 - 5 and x1 <= width + 7 + 64 + 5 (same in y without the 5).
static inline PP_HD void phase_plane_region(int width, int height, int box[4])
{
    box[0] = -PP_PAD; box[1] = width + PP_PAD;
    box[2] = -PP_PAD; box[3] = height + PP_PAD;
}
