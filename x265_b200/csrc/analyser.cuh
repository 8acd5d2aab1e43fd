// x265_b200/csrc/analyser.cuh -- host side of the frame-level CTU-analysis pipeline: geometry tables,
// device residency of the source / reference planes, and the e2e (host buffers) / resident entry points.
#pragma once
#include "common.cuh"
#include "frame.cuh"
#include "me.cuh"
#include "me_window.cuh"
#include "phase_planes.cuh"
#include <vector>
#include <stdlib.h>

struct x265cu_analyser
{
    x265cu_ctx* ctx;
    x265cu_analysis_params p;
    int stride, planeRows, fw, fh;
    size_t planeBytes, orgBytes;        // origin pixel byte offset inside a plane allocation
    int njobs, ncu, ntu; int64_t ncoef;
    // device
    uint8_t* d_fenc; uint8_t* d_refs[16]; uint8_t* d_recon[4];
    void** d_refTable; void** d_reconTable;
    int16_t* d_field; uint16_t* d_mvcost; int mvrange;
    PuDesc* d_pus; CuDesc* d_cus; TuDesc* d_tus; int32_t* d_cu_jobs;
    x265cu_me_job* d_jobs; int32_t* d_me_out; int2* d_me_packed;
    int16_t* d_coef; unsigned long long* d_cu_sse; uint32_t* d_cu_numsig; int32_t* d_cu_ref; uint32_t* d_intra;
    // pinned host staging for the e2e path
    uint8_t* h_fenc; int16_t* h_field;
    cudaEvent_t ev[5]; int ev_valid;      // stage boundaries of the last an_run (ME build+search+pack | residual | intra)
    std::vector<PuDesc> pus; std::vector<CuDesc> cus; std::vector<TuDesc> tus; std::vector<int32_t> cu_jobs;
    // first PU job / CU / TU of every CTU row (+ one past the end): the lists are in CTU raster order, so a CTU-row
    // range [r0, r1) is one contiguous slice of each list (what a WPP row shard owns, frameencoder.cpp:850-868)
    int ctuRows; std::vector<int> rowJob, rowCu, rowTu;
    // 4:2:0 chroma planes for the chroma-SATD term of subpelCompare (x265cu_analyser_enable_chroma): half resolution,
    // stride / 2 elements per row, margins = half the luma margins (picyuv.cpp:87-94)
    int chromaOn, cstride, cRows; size_t cPlaneBytes, cOrgBytes;
    uint8_t* d_fencC[2]; uint8_t* d_refC[16][2];
    void** d_refCbTable; void** d_refCrTable;
    // shared-memory-window integer search (me_window.cuh): group tables (two classes), tensor maps of the reference
    // planes [ref][MEW_NCLS], leftover list.  windowOn = 0 (X265CU_ME_WINDOW=0) keeps the global-memory kernel for all jobs.
    int windowOn; MeGroup* d_groups[3]; int32_t* d_grpJobs[3]; std::vector<int> rowGrp[3];
    CUtensorMap* d_tmaps; int32_t* d_left;
    int32_t* d_order;                     // jobs of every CTU row sorted by PU shape (geometry.h)
    // quarter-pel phase planes (phase_planes.cuh): ppOn = 0 (X265CU_ME_PHASEPLANES=0) keeps the interpolating pre-check and
    // sub-pel kernels and allocates nothing extra.  Otherwise every d_refs[r] holds 16 planes ppitch bytes apart (plane 0 =
    // the reference), rebuilt by every run of the ME stage over the box of positions its jobs can read (d_ppBox).
    int ppOn; size_t ppitch; int* d_ppBox;
    cudaEvent_t ev_pp[2]; int pp_valid;   // plane build of the last an_run
};

static const int AN_MARGIN_X = 96, AN_MARGIN_Y = 80;       // picyuv.cpp:87-88 with maxCUSize 64
// the 8-tap support (3 before, 4 after) of every phase-plane position a job can read stays inside the allocation
static_assert(PP_PAD + 3 <= AN_MARGIN_X && PP_PAD + 4 <= AN_MARGIN_Y, "phase-plane region exceeds the plane margins");

template <typename T> static T* an_upload(x265cu_ctx* c, const std::vector<T>& v)
{
    T* d = (T*)x265cu_malloc(c, v.size() * sizeof(T) + 16);
    if (d && !v.empty()) cudaMemcpy(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice);
    return d;
}

static void an_build_geometry(x265cu_analyser* a)
{
    FrameGeometry g;
    geometry_build(a->p.width, a->p.height, a->stride, a->p.numRefs, a->p.rect, a->p.amp, g);
    a->pus.swap(g.pus); a->cus.swap(g.cus); a->tus.swap(g.tus); a->cu_jobs.swap(g.cu_jobs);
    a->ctuRows = g.ctuRows; a->rowJob.swap(g.rowJob); a->rowCu.swap(g.rowCu); a->rowTu.swap(g.rowTu);
    a->njobs = (int)a->pus.size(); a->ncu = (int)a->cus.size(); a->ntu = (int)a->tus.size(); a->ncoef = g.ncoef;
    a->d_order = an_upload(a->ctx, g.order);
    for (int k = 0; k < 3; k++)
    {
        std::vector<MeGroup> grp(g.grpFirst[k].size());
        for (size_t i = 0; i < grp.size(); i++) { grp[i].first = g.grpFirst[k][i]; grp[i].count = g.grpCount[k][i]; }
        a->d_groups[k] = an_upload(a->ctx, grp);
        a->d_grpJobs[k] = an_upload(a->ctx, g.grpJobs[k]);
        a->rowGrp[k].swap(g.rowGrp[k]);
    }
}

// Runs the stages over the CTU rows [r0, r1).  Every list is sliced by pointer offset only: PU jobs, ME results and
// the intra table are indexed by the slice-local index inside the kernels, CU / TU records carry absolute indices.
static int an_run(x265cu_analyser* a, int stages, int r0, int r1)
{
    x265cu_ctx* c = a->ctx;
    const int depth = a->p.depth;
    cudaSetDevice(c->device);
    if (r0 < 0 || r1 > a->ctuRows || r0 >= r1) { x265cu_set_error("analyser: bad CTU row range", cudaErrorInvalidValue, __FILE__, __LINE__); return -1; }
    const int job0 = a->rowJob[r0], nj = a->rowJob[r1] - job0;
    const int cu0 = a->rowCu[r0], ncu = a->rowCu[r1] - cu0;
    const int tu0 = a->rowTu[r0], ntu = a->rowTu[r1] - tu0;
    a->ev_valid = stages;
    a->pp_valid = 0;
    CU_CHECK(cudaEventRecord(a->ev[0], c->stream));
    if ((stages & 1) && nj > 0)
    {
        k_build_me_jobs<<<(nj + 255) / 256, 256, 0, c->stream>>>(a->d_pus + job0, nj, a->d_field, a->fw, a->fh, a->p.width, a->p.height,
                                                                 a->stride, a->p.method, a->p.subme, a->p.merange, a->d_jobs + job0);
        CU_LAUNCH_CHECK(c);
        if (a->ppOn)
        {
            // phase planes of every reference over the positions this slice's jobs can read (a row slice builds its band only)
            CU_CHECK(cudaEventRecord(a->ev_pp[0], c->stream));
            CU_CHECK(cudaMemsetAsync(a->d_ppBox, 0x7f, sizeof(int) * 4 * 16, c->stream));       // 0x7f7f7f7f: empty box
            k_phase_plane_box<<<(nj + 255) / 256, 256, 0, c->stream>>>(a->d_jobs + job0, nj, a->stride, a->d_ppBox);
            CU_LAUNCH_CHECK(c);
            int reg[4];
            phase_plane_region(a->p.width, a->p.height, reg);
            const dim3 grid((reg[1] - reg[0] + PP_TW - 1) / PP_TW, (reg[3] - reg[2] + PP_TH - 1) / PP_TH, a->p.numRefs);
            const int lastX = a->stride - AN_MARGIN_X - 1, lastY = a->planeRows - AN_MARGIN_Y - 1;
            if (depth == 8) k_luma_phase_planes<uint8_t><<<grid, 256, 0, c->stream>>>((uint8_t* const*)a->d_refTable, a->stride, a->ppitch, a->d_ppBox, reg[1], reg[3], lastX, lastY);
            else            k_luma_phase_planes<uint16_t><<<grid, 256, 0, c->stream>>>((uint8_t* const*)a->d_refTable, a->stride, a->ppitch, a->d_ppBox, reg[1], reg[3], lastX, lastY);
            CU_LAUNCH_CHECK(c);
            CU_CHECK(cudaEventRecord(a->ev_pp[1], c->stream));
            a->pp_valid = 1;
        }
        MeChromaArgs ch;
        if (a->chromaOn)
        {
            ch.fencCb = a->d_fencC[0] + a->cOrgBytes; ch.fencCr = a->d_fencC[1] + a->cOrgBytes;
            ch.refCb = (const void* const*)a->d_refCbTable; ch.refCr = (const void* const*)a->d_refCrTable; ch.cstride = a->cstride;
        }
        MeWinLaunch win;
        if (a->windowOn)
        {
            win.tmaps = a->d_tmaps; win.allocX = AN_MARGIN_X; win.allocY = AN_MARGIN_Y;
            win.amp = a->p.amp;
            for (int k = 0; k < 3; k++)
            {
                win.groups[k] = a->d_groups[k] + a->rowGrp[k][r0]; win.ngroups[k] = a->rowGrp[k][r1] - a->rowGrp[k][r0];
                win.grp_jobs[k] = a->d_grpJobs[k];
            }
            win.job0 = job0; win.left_count = c->d_counter + 9; win.left_list = a->d_left;
            win.order = a->d_order + job0;
        }
        if (launch_me(c, depth, a->d_fenc + a->orgBytes, a->stride, (const void* const*)a->d_refTable, a->stride, 0,
                      a->d_mvcost + a->mvrange, a->d_jobs + job0, nj, a->d_me_out + (size_t)job0 * 4, c->d_counter,
                      a->chromaOn ? &ch : NULL, a->windowOn ? &win : NULL, a->ppOn ? (int)a->ppitch : 0)) return -1;
        CU_CHECK(cudaEventRecord(a->ev[4], c->stream));      // ME search kernel alone ends here
        k_pack_me<<<(nj + 255) / 256, 256, 0, c->stream>>>(a->d_me_out + (size_t)job0 * 4, nj, a->d_me_packed + job0);
        CU_LAUNCH_CHECK(c);
    }
    else if (stages & 1) CU_CHECK(cudaEventRecord(a->ev[4], c->stream));
    CU_CHECK(cudaEventRecord(a->ev[1], c->stream));
    if ((stages & 2) && ntu > 0)
    {
        CU_CHECK(cudaMemsetAsync(a->d_cu_sse + cu0, 0, sizeof(unsigned long long) * ncu, c->stream));
        CU_CHECK(cudaMemsetAsync(a->d_cu_numsig + cu0, 0, sizeof(uint32_t) * ncu, c->stream));
        int blocks = ntu < c->sm_count * 8 ? ntu : c->sm_count * 8;
        if (depth == 8)
            k_cu_residual<uint8_t><<<blocks, 256, 0, c->stream>>>((const uint8_t*)(a->d_fenc + a->orgBytes), (const uint8_t* const*)a->d_refTable, a->stride,
                a->d_cus, a->d_tus + tu0, ntu, a->d_cu_jobs, a->p.numRefs, a->d_me_out, a->p.qp, a->d_coef, (uint8_t* const*)a->d_reconTable,
                a->d_cu_sse, a->d_cu_numsig, a->d_cu_ref);
        else
            k_cu_residual<uint16_t><<<blocks, 256, 0, c->stream>>>((const uint16_t*)(a->d_fenc + a->orgBytes), (const uint16_t* const*)a->d_refTable, a->stride,
                a->d_cus, a->d_tus + tu0, ntu, a->d_cu_jobs, a->p.numRefs, a->d_me_out, a->p.qp, a->d_coef, (uint16_t* const*)a->d_reconTable,
                a->d_cu_sse, a->d_cu_numsig, a->d_cu_ref);
        CU_LAUNCH_CHECK(c);
    }
    CU_CHECK(cudaEventRecord(a->ev[2], c->stream));
    if ((stages & 4) && ncu > 0)
    {
        int blocks = ncu < c->sm_count * 8 ? ncu : c->sm_count * 8;
        if (depth == 8) k_intra_search<uint8_t><<<blocks, 256, 0, c->stream>>>((const uint8_t*)(a->d_fenc + a->orgBytes), a->stride, a->d_cus + cu0, ncu, a->d_intra + (size_t)cu0 * 36);
        else            k_intra_search<uint16_t><<<blocks, 256, 0, c->stream>>>((const uint16_t*)(a->d_fenc + a->orgBytes), a->stride, a->d_cus + cu0, ncu, a->d_intra + (size_t)cu0 * 36);
        CU_LAUNCH_CHECK(c);
    }
    CU_CHECK(cudaEventRecord(a->ev[3], c->stream));
    return 0;
}

// upload a width x height host image into a margin-extended device plane
static int an_upload_plane(x265cu_analyser* a, uint8_t* d_plane, const void* host, int hostStride)
{
    x265cu_ctx* c = a->ctx;
    const size_t es = a->p.depth == 8 ? 1 : 2;
    cudaSetDevice(c->device);
    CU_CHECK(cudaMemcpy2DAsync(d_plane + a->orgBytes, (size_t)a->stride * es, host, (size_t)hostStride * es,
                               (size_t)a->p.width * es, a->p.height, cudaMemcpyHostToDevice, c->stream));
    return x265cu_extend_border(c, a->p.depth, d_plane + a->orgBytes, a->stride, a->p.width, a->p.height, AN_MARGIN_X, AN_MARGIN_Y);
}

extern "C" {

x265cu_analyser* x265cu_analyser_create(x265cu_ctx* ctx, const x265cu_analysis_params* p)
{
    if (!ctx || p->numRefs < 1 || p->numRefs > 16 || (p->depth != 8 && p->depth != 10)) return NULL;
    cudaSetDevice(ctx->device);
    x265cu_analyser* a = new x265cu_analyser();
    a->ctx = ctx; a->p = *p;
    const size_t es = p->depth == 8 ? 1 : 2;
    a->stride = (p->width + 2 * AN_MARGIN_X + 63) / 64 * 64;
    a->planeRows = p->height + 2 * AN_MARGIN_Y;
    a->planeBytes = (size_t)a->stride * a->planeRows * es + 256;
    a->orgBytes = ((size_t)AN_MARGIN_Y * a->stride + AN_MARGIN_X) * es;
    a->fw = (p->width + 15) / 16; a->fh = (p->height + 15) / 16;
    an_build_geometry(a);
    a->d_fenc = (uint8_t*)x265cu_malloc(ctx, a->planeBytes);
    if (a->d_fenc) cudaMemset(a->d_fenc, 0, a->planeBytes);
    // quarter-pel phase planes: 16 planes per reference allocation.  The ME kernels address a candidate by an int byte offset
    // from its PU's origin in plane 0, which must reach the last plane's last row.
    {
        const char* e = getenv("X265CU_ME_PHASEPLANES");
        a->ppOn = !(e && e[0] == '0');
        a->ppitch = (a->planeBytes + 255) / 256 * 256;
        if (a->ppOn && 16 * a->ppitch > (size_t)INT_MAX)
        {
            x265cu_set_error("analyser: phase planes do not fit int byte offsets (set X265CU_ME_PHASEPLANES=0)", cudaErrorInvalidValue, __FILE__, __LINE__);
            delete a;
            return NULL;
        }
    }
    const size_t refBytes = a->ppOn ? 16 * a->ppitch : a->planeBytes;
    void* reft[16]; void* rect[4];
    for (int r = 0; r < p->numRefs; r++) { a->d_refs[r] = (uint8_t*)x265cu_malloc(ctx, refBytes); if (a->d_refs[r]) cudaMemset(a->d_refs[r], 0, refBytes); reft[r] = a->d_refs[r] + a->orgBytes; }
    a->d_ppBox = a->ppOn ? (int*)x265cu_malloc(ctx, sizeof(int) * 4 * 16) : NULL;
    for (int d = 0; d < 4; d++) { a->d_recon[d] = (uint8_t*)x265cu_malloc(ctx, a->planeBytes); rect[d] = a->d_recon[d] + a->orgBytes; cudaMemset(a->d_recon[d], 0, a->planeBytes); }
    a->d_refTable = (void**)x265cu_malloc(ctx, sizeof(void*) * 16);
    a->d_reconTable = (void**)x265cu_malloc(ctx, sizeof(void*) * 4);
    cudaMemcpy(a->d_refTable, reft, sizeof(void*) * p->numRefs, cudaMemcpyHostToDevice);
    cudaMemcpy(a->d_reconTable, rect, sizeof(void*) * 4, cudaMemcpyHostToDevice);
    const size_t fieldBytes = (size_t)p->numRefs * a->fw * a->fh * 2 * sizeof(int16_t);
    a->d_field = (int16_t*)x265cu_malloc(ctx, fieldBytes);
    a->mvrange = 65536;                                   // +-2*BC_MAX_MV like bitcost.h:77
    std::vector<uint16_t> tab(2 * a->mvrange + 1);
    x265cu_mvcost_table(p->lambda, a->mvrange, tab.data());
    a->d_mvcost = an_upload(ctx, tab);
    a->d_pus = an_upload(ctx, a->pus); a->d_cus = an_upload(ctx, a->cus); a->d_tus = an_upload(ctx, a->tus); a->d_cu_jobs = an_upload(ctx, a->cu_jobs);
    a->d_jobs = (x265cu_me_job*)x265cu_malloc(ctx, sizeof(x265cu_me_job) * a->njobs);
    a->d_me_out = (int32_t*)x265cu_malloc(ctx, sizeof(int32_t) * 4 * a->njobs);
    a->d_me_packed = (int2*)x265cu_malloc(ctx, sizeof(int2) * a->njobs);
    // shared-memory-window search: tensor maps over the reference plane allocations (STAR only; the other methods and any
    // group whose window does not fit go through the global-memory kernel)
    {
        const char* e = getenv("X265CU_ME_WINDOW");
        a->windowOn = !(e && e[0] == '0') && p->method == 3;
        a->d_tmaps = NULL;
        a->d_left = (int32_t*)x265cu_malloc(ctx, sizeof(int32_t) * (a->njobs + 1));
        if (a->windowOn)
        {
            std::vector<CUtensorMap> tm((size_t)p->numRefs * MEW_NCLS);
            bool ok = a->d_left != NULL;
            for (int r = 0; r < p->numRefs && ok; r++)
                ok = a->d_refs[r] && mew_build_tmaps(a->d_refs[r], a->stride, a->planeRows, (int)es, &tm[(size_t)r * MEW_NCLS]) == 0;
            if (ok)
            {
                a->d_tmaps = (CUtensorMap*)x265cu_malloc(ctx, sizeof(CUtensorMap) * tm.size());
                ok = a->d_tmaps && cudaMemcpy(a->d_tmaps, tm.data(), sizeof(CUtensorMap) * tm.size(), cudaMemcpyHostToDevice) == cudaSuccess;
            }
            if (!ok) { fprintf(stderr, "x265cu: tensor maps unavailable, integer search stays on the global-memory kernel: %s\n", x265cu_last_error()); a->windowOn = 0; }
        }
    }
    a->d_coef = (int16_t*)x265cu_malloc(ctx, sizeof(int16_t) * a->ncoef);
    a->d_cu_sse = (unsigned long long*)x265cu_malloc(ctx, sizeof(unsigned long long) * a->ncu);
    a->d_cu_numsig = (uint32_t*)x265cu_malloc(ctx, sizeof(uint32_t) * a->ncu);
    a->d_cu_ref = (int32_t*)x265cu_malloc(ctx, sizeof(int32_t) * a->ncu);
    a->d_intra = (uint32_t*)x265cu_malloc(ctx, sizeof(uint32_t) * 36 * a->ncu);
    for (int i = 0; i < 5; i++) cudaEventCreate(&a->ev[i]);
    for (int i = 0; i < 2; i++) cudaEventCreate(&a->ev_pp[i]);
    a->ev_valid = 0; a->pp_valid = 0;
    a->chromaOn = 0; a->d_refCbTable = a->d_refCrTable = NULL;
    a->d_fencC[0] = a->d_fencC[1] = NULL;
    for (int r = 0; r < 16; r++) a->d_refC[r][0] = a->d_refC[r][1] = NULL;
    a->h_fenc = (uint8_t*)x265cu_host_alloc((size_t)p->width * p->height * es);
    a->h_field = (int16_t*)x265cu_host_alloc(fieldBytes);
    if (!a->d_intra || !a->d_coef || !a->d_me_out || !a->h_fenc || !a->h_field || (a->ppOn && !a->d_ppBox)) return NULL;
    cudaDeviceSynchronize();
    return a;
}

void x265cu_analyser_destroy(x265cu_analyser* a)
{
    if (!a) return;
    x265cu_ctx* c = a->ctx;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    void* bufs[] = { a->d_fenc, a->d_refTable, a->d_reconTable, a->d_field, a->d_mvcost, a->d_pus, a->d_cus, a->d_tus, a->d_cu_jobs, a->d_jobs,
                     a->d_me_out, a->d_me_packed, a->d_coef, a->d_cu_sse, a->d_cu_numsig, a->d_cu_ref, a->d_intra,
                     a->d_groups[0], a->d_groups[1], a->d_groups[2], a->d_grpJobs[0], a->d_grpJobs[1], a->d_grpJobs[2], a->d_tmaps, a->d_left, a->d_order,
                     a->d_ppBox };
    for (void* b : bufs) cudaFree(b);
    for (int r = 0; r < a->p.numRefs; r++) cudaFree(a->d_refs[r]);
    for (int d = 0; d < 4; d++) cudaFree(a->d_recon[d]);
    for (int k = 0; k < 2; k++) { cudaFree(a->d_fencC[k]); for (int r = 0; r < a->p.numRefs; r++) cudaFree(a->d_refC[r][k]); }
    cudaFree(a->d_refCbTable); cudaFree(a->d_refCrTable);
    x265cu_host_free(a->h_fenc); x265cu_host_free(a->h_field);
    for (int i = 0; i < 5; i++) cudaEventDestroy(a->ev[i]);
    for (int i = 0; i < 2; i++) cudaEventDestroy(a->ev_pp[i]);
    delete a;
}

int x265cu_analyser_counts(x265cu_analyser* a, int* njobs, int* ncu, int* ntu, int64_t* ncoef, int* stride)
{
    *njobs = a->njobs; *ncu = a->ncu; *ntu = a->ntu; *ncoef = a->ncoef; *stride = a->stride;
    return 0;
}

int x265cu_analyser_set_ref(x265cu_analyser* a, int idx, const void* host_luma, int host_stride)
{
    if (idx < 0 || idx >= a->p.numRefs) return -1;
    if (an_upload_plane(a, a->d_refs[idx], host_luma, host_stride)) return -1;
    return x265cu_sync(a->ctx);
}

int x265cu_analyser_load_inputs(x265cu_analyser* a, const void* fenc_host, int host_stride, const int16_t* field_host)
{
    x265cu_ctx* c = a->ctx;
    const size_t es = a->p.depth == 8 ? 1 : 2;
    // copies are issued straight from the caller's buffers: pass pinned memory (x265cu_host_alloc)
    // for true asynchronous DMA; pageable memory also works (the driver stages it)
    (void)es;
    const size_t fieldBytes = (size_t)a->p.numRefs * a->fw * a->fh * 2 * sizeof(int16_t);
    if (an_upload_plane(a, a->d_fenc, fenc_host, host_stride)) return -1;
    CU_CHECK(cudaMemcpyAsync(a->d_field, field_host, fieldBytes, cudaMemcpyHostToDevice, c->stream));
    return 0;
}

// ---- 4:2:0 chroma for the chroma-SATD term of subpelCompare (MotionEstimate::bChromaSATD, motion.cpp:204-212, 1601-1661) ----
// After enable_chroma() the ME stage runs the k_me_chroma launches (x265cu_me_batch_chroma's kernels) on the resident chroma
// planes; the caller uploads the source's Cb / Cr with load_chroma() and every reference's with set_ref_chroma().
static int an_upload_cplane(x265cu_analyser* a, uint8_t* d_plane, const void* host, int hostStride)
{
    x265cu_ctx* c = a->ctx;
    const size_t es = a->p.depth == 8 ? 1 : 2;
    const int cw = a->p.width >> 1, ch = a->p.height >> 1;
    cudaSetDevice(c->device);
    CU_CHECK(cudaMemcpy2DAsync(d_plane + a->cOrgBytes, (size_t)a->cstride * es, host, (size_t)hostStride * es,
                               (size_t)cw * es, ch, cudaMemcpyHostToDevice, c->stream));
    return x265cu_extend_border(c, a->p.depth, d_plane + a->cOrgBytes, a->cstride, cw, ch, AN_MARGIN_X / 2, AN_MARGIN_Y / 2);
}

int x265cu_analyser_enable_chroma(x265cu_analyser* a)
{
    if (a->chromaOn) return 0;
    x265cu_ctx* c = a->ctx;
    cudaSetDevice(c->device);
    const size_t es = a->p.depth == 8 ? 1 : 2;
    a->cstride = a->stride / 2;
    a->cRows = (a->p.height >> 1) + AN_MARGIN_Y;                 // 2 * (AN_MARGIN_Y / 2)
    a->cPlaneBytes = (size_t)a->cstride * a->cRows * es + 256;
    a->cOrgBytes = ((size_t)(AN_MARGIN_Y / 2) * a->cstride + AN_MARGIN_X / 2) * es;
    void* cbt[16]; void* crt[16];
    for (int k = 0; k < 2; k++)
    {
        a->d_fencC[k] = (uint8_t*)x265cu_malloc(c, a->cPlaneBytes);
        if (!a->d_fencC[k]) return -1;
        CU_CHECK(cudaMemset(a->d_fencC[k], 0, a->cPlaneBytes));
        for (int r = 0; r < a->p.numRefs; r++)
        {
            a->d_refC[r][k] = (uint8_t*)x265cu_malloc(c, a->cPlaneBytes);
            if (!a->d_refC[r][k]) return -1;
            CU_CHECK(cudaMemset(a->d_refC[r][k], 0, a->cPlaneBytes));
            (k ? crt : cbt)[r] = a->d_refC[r][k] + a->cOrgBytes;
        }
    }
    a->d_refCbTable = (void**)x265cu_malloc(c, sizeof(void*) * 16);
    a->d_refCrTable = (void**)x265cu_malloc(c, sizeof(void*) * 16);
    if (!a->d_refCbTable || !a->d_refCrTable) return -1;
    CU_CHECK(cudaMemcpy(a->d_refCbTable, cbt, sizeof(void*) * a->p.numRefs, cudaMemcpyHostToDevice));
    CU_CHECK(cudaMemcpy(a->d_refCrTable, crt, sizeof(void*) * a->p.numRefs, cudaMemcpyHostToDevice));
    a->chromaOn = 1;
    return 0;
}

int x265cu_analyser_set_ref_chroma(x265cu_analyser* a, int idx, const void* cb_host, const void* cr_host, int host_stride)
{
    if (!a->chromaOn || idx < 0 || idx >= a->p.numRefs) return -1;
    if (an_upload_cplane(a, a->d_refC[idx][0], cb_host, host_stride) || an_upload_cplane(a, a->d_refC[idx][1], cr_host, host_stride)) return -1;
    return x265cu_sync(a->ctx);
}

int x265cu_analyser_load_chroma(x265cu_analyser* a, const void* cb_host, const void* cr_host, int host_stride)
{
    if (!a->chromaOn) return -1;
    if (an_upload_cplane(a, a->d_fencC[0], cb_host, host_stride) || an_upload_cplane(a, a->d_fencC[1], cr_host, host_stride)) return -1;
    return 0;
}

int x265cu_analyser_run_resident(x265cu_analyser* a, int stages) { return an_run(a, stages, 0, a->ctuRows); }

// ---- CTU-row shards (the WPP row partition of SURVEY 8(e): frameencoder.cpp:850-868 enables row r once the
// reference rows it needs are reconstructed; a rank owns a set of CTU rows and analyses exactly those) ----
int x265cu_analyser_ctu_rows(x265cu_analyser* a) { return a->ctuRows; }

int x265cu_analyser_row_range(x265cu_analyser* a, int ctuRow0, int ctuRow1, int* job0, int* njobs, int* cu0, int* ncu)
{
    if (ctuRow0 < 0 || ctuRow1 > a->ctuRows || ctuRow0 > ctuRow1) return -1;
    *job0 = a->rowJob[ctuRow0]; *njobs = a->rowJob[ctuRow1] - a->rowJob[ctuRow0];
    *cu0 = a->rowCu[ctuRow0];   *ncu = a->rowCu[ctuRow1] - a->rowCu[ctuRow0];
    return 0;
}

int x265cu_analyser_run_rows(x265cu_analyser* a, int stages, int ctuRow0, int ctuRow1) { return an_run(a, stages, ctuRow0, ctuRow1); }

// `out` arrays are always full-frame sized; a row shard fills only the entries of its own rows.
int x265cu_analyser_analyse_rows(x265cu_analyser* a, const void* fenc_host, int host_stride, const int16_t* field_host, int stages,
                                 int ctuRow0, int ctuRow1, x265cu_analysis_out* out)
{
    x265cu_ctx* c = a->ctx;
    if (x265cu_analyser_load_inputs(a, fenc_host, host_stride, field_host)) return -1;
    if (an_run(a, stages, ctuRow0, ctuRow1)) return -1;
    if (out)
    {
        const size_t j0 = a->rowJob[ctuRow0], nj = a->rowJob[ctuRow1] - j0, c0 = a->rowCu[ctuRow0], nc = a->rowCu[ctuRow1] - c0;
        if (out->me_packed && nj) CU_CHECK(cudaMemcpyAsync(out->me_packed + 2 * j0, a->d_me_packed + j0, sizeof(int2) * nj, cudaMemcpyDeviceToHost, c->stream));
        if (out->cu_sse && nc) CU_CHECK(cudaMemcpyAsync(out->cu_sse + c0, a->d_cu_sse + c0, sizeof(uint64_t) * nc, cudaMemcpyDeviceToHost, c->stream));
        if (out->cu_numsig && nc) CU_CHECK(cudaMemcpyAsync(out->cu_numsig + c0, a->d_cu_numsig + c0, sizeof(uint32_t) * nc, cudaMemcpyDeviceToHost, c->stream));
        if (out->cu_ref && nc) CU_CHECK(cudaMemcpyAsync(out->cu_ref + c0, a->d_cu_ref + c0, sizeof(int32_t) * nc, cudaMemcpyDeviceToHost, c->stream));
        if (out->intra_cost && nc) CU_CHECK(cudaMemcpyAsync(out->intra_cost + 36 * c0, a->d_intra + 36 * c0, sizeof(uint32_t) * 36 * nc, cudaMemcpyDeviceToHost, c->stream));
    }
    CU_CHECK(cudaStreamSynchronize(c->stream));
    return 0;
}

int x265cu_analyser_analyse(x265cu_analyser* a, const void* fenc_host, int host_stride, const int16_t* field_host, int stages,
                            x265cu_analysis_out* out)
{
    return x265cu_analyser_analyse_rows(a, fenc_host, host_stride, field_host, stages, 0, a->ctuRows, out);
}

// per-stage device time of the last run (ms): [0] ME stage (job build + search + pack), [1] residual,
// [2] intra, [3] the ME search kernel alone.  Synchronises the stream.
int x265cu_analyser_stage_ms(x265cu_analyser* a, float* ms)
{
    CU_CHECK(cudaEventSynchronize(a->ev[3]));
    for (int i = 0; i < 3; i++) CU_CHECK(cudaEventElapsedTime(&ms[i], a->ev[i], a->ev[i + 1]));
    ms[3] = 0.f;
    if (a->ev_valid & 1) CU_CHECK(cudaEventElapsedTime(&ms[3], a->ev[0], a->ev[4]));
    return 0;
}

// device time (ms) of the phase-plane build of the last run (0 when it built none: planes off, or no ME stage).
// Synchronises on it.  It lies inside stage_ms()[0].
int x265cu_analyser_phase_planes_ms(x265cu_analyser* a, float* ms)
{
    *ms = 0.f;
    if (!a->pp_valid) return 0;
    CU_CHECK(cudaEventSynchronize(a->ev_pp[1]));
    CU_CHECK(cudaEventElapsedTime(ms, a->ev_pp[0], a->ev_pp[1]));
    return 0;
}

// device address of pixel (0, 0) of reference idx's quarter-pel phase plane `phase` = (yFrac << 2) | xFrac (0 = the
// reference itself; same stride as x265cu_analyser_ref_plane).  NULL for phase > 0 when the planes are off.
void* x265cu_analyser_ref_plane_phase(x265cu_analyser* a, int idx, int phase)
{
    if (idx < 0 || idx >= a->p.numRefs || phase < 0 || phase > 15 || (phase && !a->ppOn)) return NULL;
    return a->d_refs[idx] + (size_t)phase * a->ppitch + a->orgBytes;
}

// the rectangle [box[0], box[1]) x [box[2], box[3]) (picture pixels) of reference idx's phase planes that the last run
// built: the union of its jobs' read boxes (phase_planes.h) clipped to phase_plane_region(); empty (x0 >= x1) when
// none.  Synchronises the stream.
int x265cu_analyser_phase_region(x265cu_analyser* a, int idx, int* box)
{
    if (idx < 0 || idx >= a->p.numRefs || !a->ppOn) return -1;
    int b[4], reg[4];
    cudaSetDevice(a->ctx->device);
    CU_CHECK(cudaMemcpyAsync(b, a->d_ppBox + 4 * idx, sizeof(b), cudaMemcpyDeviceToHost, a->ctx->stream));
    CU_CHECK(cudaStreamSynchronize(a->ctx->stream));
    phase_plane_region(a->p.width, a->p.height, reg);
    box[0] = b[0] > reg[0] ? b[0] : reg[0]; box[1] = -b[1] < reg[1] ? -b[1] : reg[1];
    box[2] = b[2] > reg[2] ? b[2] : reg[2]; box[3] = -b[3] < reg[3] ? -b[3] : reg[3];
    return 0;
}

// device address of reference plane idx's origin pixel and the plane geometry, so that the owner of the
// reconstructed pixels (e.g. an NCCL broadcast) can write them in place; call x265cu_analyser_ref_updated()
// afterwards to re-extend the borders.
void* x265cu_analyser_ref_plane(x265cu_analyser* a, int idx, int* stride)
{
    if (idx < 0 || idx >= a->p.numRefs) return NULL;
    *stride = a->stride;
    return a->d_refs[idx] + a->orgBytes;
}
int x265cu_analyser_ref_updated(x265cu_analyser* a, int idx)
{
    if (idx < 0 || idx >= a->p.numRefs) return -1;
    cudaSetDevice(a->ctx->device);
    return x265cu_extend_border(a->ctx, a->p.depth, a->d_refs[idx] + a->orgBytes, a->stride, a->p.width, a->p.height, AN_MARGIN_X, AN_MARGIN_Y);
}

// device address of the origin pixel of reconstruction plane `depthIdx` (0..3 = CU size 64, 32, 16, 8): what a row
// shard's owner broadcasts (the producer side of m_reconRowFlag, framefilter.cpp:664)
void* x265cu_analyser_recon_plane(x265cu_analyser* a, int depthIdx, int* stride)
{
    if (depthIdx < 0 || depthIdx >= 4) return NULL;
    *stride = a->stride;
    return a->d_recon[depthIdx] + a->orgBytes;
}
// promote the reconstructed CTU rows [ctuRow0, ctuRow1) of recon plane depthIdx to reference idx (device copy);
// call x265cu_analyser_ref_updated() once all rows of the new reference are in place
int x265cu_analyser_recon_to_ref(x265cu_analyser* a, int depthIdx, int idx, int ctuRow0, int ctuRow1)
{
    if (depthIdx < 0 || depthIdx >= 4 || idx < 0 || idx >= a->p.numRefs || ctuRow0 < 0 || ctuRow1 > a->ctuRows || ctuRow0 >= ctuRow1) return -1;
    const size_t es = a->p.depth == 8 ? 1 : 2;
    const int y0 = ctuRow0 * 64, y1 = ctuRow1 * 64 < a->p.height ? ctuRow1 * 64 : a->p.height;
    cudaSetDevice(a->ctx->device);
    const size_t off = a->orgBytes + (size_t)y0 * a->stride * es, pitch = (size_t)a->stride * es;
    CU_CHECK(cudaMemcpy2DAsync(a->d_refs[idx] + off, pitch, a->d_recon[depthIdx] + off, pitch, (size_t)a->p.width * es, y1 - y0,
                               cudaMemcpyDeviceToDevice, a->ctx->stream));
    return 0;
}

// debugging / parity access to device-resident results
int x265cu_analyser_fetch(x265cu_analyser* a, int what, void* host)
{
    x265cu_ctx* c = a->ctx;
    const size_t es = a->p.depth == 8 ? 1 : 2;
    const void* src = NULL; size_t bytes = 0;
    cudaSetDevice(c->device);
    switch (what)
    {
    case 0: src = a->d_jobs; bytes = sizeof(x265cu_me_job) * a->njobs; break;
    case 1: src = a->d_me_out; bytes = sizeof(int32_t) * 4 * a->njobs; break;
    case 2: src = a->d_coef; bytes = sizeof(int16_t) * a->ncoef; break;
    case 3: case 4: case 5: case 6: src = a->d_recon[what - 3]; bytes = (size_t)a->stride * a->planeRows * es; break;
    case 7: src = a->d_cu_jobs; bytes = sizeof(int32_t) * a->ncu * a->p.numRefs; break;
    case 8: src = a->d_fenc; bytes = (size_t)a->stride * a->planeRows * es; break;
    default: return -1;
    }
    CU_CHECK(cudaMemcpyAsync(host, src, bytes, cudaMemcpyDeviceToHost, c->stream));
    CU_CHECK(cudaStreamSynchronize(c->stream));
    return 0;
}

} // extern "C"
