// tests/phase_planes_capi.cpp -- CPU-only test shim: exposes the phase-plane bound arithmetic
// (x265_b200/csrc/phase_planes.h, the code the frame analyser's plane build runs) to tests/test_gpu_phase_planes.py.
#include "../x265_b200/csrc/phase_planes.h"
#include <stdint.h>

extern "C" {

int pp_pad(void) { return PP_PAD; }

void pp_region(int width, int height, int* box) { phase_plane_region(width, height, box); }

// box of every job: jobs = n x 8 int32 {x, y, w, h, minx, miny, maxx, maxy}, boxes = n x 4 int32 {x0, x1, y0, y1}
void pp_job_boxes(const int32_t* jobs, int n, int32_t* boxes)
{
    for (int i = 0; i < n; i++)
    {
        const int32_t* j = jobs + 8 * i;
        int b[4];
        phase_plane_job_box(j[0], j[1], j[2], j[3], j[4], j[5], j[6], j[7], b);
        for (int k = 0; k < 4; k++) boxes[4 * i + k] = b[k];
    }
}

}
