/* include/x265_b200.h -- C ABI of libx265cu.so, the B200-native (sm_100a) implementation of x265's
 * block-primitive hot path.  Plain C: pointers and sizes only, no CUDA/torch types.
 *
 * Two levels, both replacing entries of the reference's EncoderPrimitives table
 * (/root/reference/source/common/primitives.h:237-429):
 *
 *  (1) PER-CALL TABLE  -- x265cu_get_primitive() hands out C function pointers with EXACTLY the
 *      reference typedefs (primitives.h:133-234): host pointers, strides in elements, caller-owned
 *      buffers, outputs fully overwritten, nothing retained.  setupCudaPrimitives() (the drop-in
 *      sibling of setupAssemblyPrimitives(), primitives.h:470, call site primitives.cpp:260-265)
 *      fills an EncoderPrimitives from these; see INTEGRATION.md.  Each call stages the block to the
 *      device, runs the same kernels as (2) with a batch of one, and copies the result back.
 *
 *  (2) BATCHED API     -- one launch per primitive class over a job list (all candidates x all CTUs
 *      of a frame / row), on device-resident planes.  This is what the batching hooks at
 *      CostEstimateGroup::finishBatch (slicetype.cpp:1942-2009) and FrameEncoder::processRowEncoder
 *      (frameencoder.cpp:1340) call.  `_dev` arguments are device pointers obtained from
 *      x265cu_malloc(); every function returns 0 on success, -1 on a CUDA error (message via
 *      x265cu_last_error()); there is NO CPU fallback.
 *
 * depth is 8 (pixel = uint8_t) or 10 (pixel = uint16_t), cf. common/common.h:126-148.
 */
#ifndef X265_B200_H
#define X265_B200_H
#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct x265cu_ctx x265cu_ctx;

/* ---------- context / memory ---------- */
int  x265cu_device_count(void);
x265cu_ctx* x265cu_create(int device);                 /* NULL if no CUDA device (never falls back) */
void x265cu_destroy(x265cu_ctx*);
const char* x265cu_last_error(void);
int  x265cu_sync(x265cu_ctx*);
void* x265cu_stream(x265cu_ctx*);                       /* cudaStream_t the ctx launches on */
void* x265cu_malloc(x265cu_ctx*, size_t bytes);
void  x265cu_free(x265cu_ctx*, void* dev);
void* x265cu_host_alloc(size_t bytes);                  /* pinned host memory */
void  x265cu_host_free(void* p);
int  x265cu_h2d(x265cu_ctx*, void* dev, const void* host, size_t bytes);   /* async on ctx stream */
int  x265cu_d2h(x265cu_ctx*, void* host, const void* dev, size_t bytes);   /* async on ctx stream */
int  x265cu_memset(x265cu_ctx*, void* dev, int value, size_t bytes);
/* strided 2-D copy on the context's stream (asynchronous): kind 0 = host->device, 1 = device->host, 2 = device->device */
int  x265cu_copy2d(x265cu_ctx*, void* dst, size_t dpitch, const void* src, size_t spitch, size_t widthBytes, size_t rows, int kind);
/* timing on the ctx stream (cudaEvent): returns ms between begin/end, <0 on error */
int  x265cu_timer_begin(x265cu_ctx*);
float x265cu_timer_end(x265cu_ctx*);
/* number of kernels this library has launched since the ctx was created */
uint64_t x265cu_launch_count(x265cu_ctx*);   /* kernel launches of the whole process so far (all contexts, per-call table included) */
/* device ms of the three launches of the last motion-estimation batch: pre-checks, integer search, sub-pel */
int x265cu_me_phase_ms(x265cu_ctx*, float ms[3]);

/* ---------- (1) per-call table ---------- */
/* name / i / j / k exactly as the fields of EncoderPrimitives: "pu.sad" (i = LumaPU),
 * "cu.dct" (i = LumaCU), "cu.intra_pred" (i = LumaCU, j = mode), "quant",
 * "chroma.pu.filter_hpp" (k = csp, i = LumaPU) ...  Returns NULL for entries we do not provide. */
void* x265cu_get_primitive(int depth, const char* name, int i, int j, int k);
/* Error convention of the per-call table (SURVEY 8b): the reference's primitives are void / value-returning and cannot
 * fail, so a CUDA failure inside a thunk never kills the process: the thunk logs, returns zeros and latches this flag.
 * The encoder-side hook polls it after x265_encoder_encode() and sets m_aborted (encoder/api.cpp:179-180, 222-229), so the
 * next x265_encoder_encode() returns < 0.  X265CU_DEVICE (environment) selects the GPU of the per-call table. */
int x265cu_primitive_error(void);
const char* x265cu_primitive_error_string(void);
void x265cu_primitive_error_clear(void);
uint64_t x265cu_primitive_calls(void);     /* per-call table invocations of this process so far (diagnostics) */

/* ---------- (2) batched API ---------- */

/* pixel-compare class: sad / satd / sa8d / sse / var / psy   (pixel.cpp:40-377, 167-186, 703-757) */
enum { X265CU_SAD = 0, X265CU_SATD = 1, X265CU_SA8D = 2, X265CU_SSE_PP = 3, X265CU_SSE_SS = 4,
       X265CU_SSD_S = 5, X265CU_VAR = 6, X265CU_PSY = 7 };
typedef struct {
    int64_t a_off, b_off;      /* element offsets into plane A / plane B */
    int32_t a_stride, b_stride;
    int16_t w, h;
    int32_t pad;
} x265cu_cmp_job;
/* out_dev[n] : uint64 (sse_t / var packing as in the reference; int costs zero-extended) */
int x265cu_pixelcmp_batch(x265cu_ctx*, int depth, int op, const void* planeA_dev, const void* planeB_dev,
                          const x265cu_cmp_job* jobs_dev, int n, uint64_t* out_dev);
/* Same costs over a regular grid: block (bx,by) compares A + by*bh*a_stride + bx*bw with the same
 * offset from B (the displacement of a whole-frame compare is baked into B); strides in pixels;
 * op = SAD / SATD / SA8D / SSE_PP; out_dev[by*nbx + bx].  This is the shape of the frame-level cost
 * passes (lowres SATD maps, slicetype.cpp:640-700; weightp cost, slicetype.cpp:462-520): no job list,
 * one lane per 16-byte column so plane reads are fully coalesced. */
int x265cu_pixelcmp_grid(x265cu_ctx*, int depth, int op, const void* A_dev, int64_t a_stride, const void* B_dev, int64_t b_stride,
                         int bw, int bh, int nbx, int nby, uint64_t* out_dev);

/* elementwise block-op class (pixel.cpp:379-862, ipfilter.cpp:40-57) */
enum { X265CU_COPY_PP = 0, X265CU_COPY_SS, X265CU_COPY_SP, X265CU_COPY_PS, X265CU_SUB_PS, X265CU_ADD_PS,
       X265CU_PIXELAVG_PP, X265CU_ADDAVG, X265CU_P2S, X265CU_TRANSPOSE, X265CU_BLOCKFILL_S,
       X265CU_CPY2DTO1D_SHL, X265CU_CPY2DTO1D_SHR, X265CU_CPY1DTO2D_SHL, X265CU_CPY1DTO2D_SHR,
       X265CU_WEIGHT_PP, X265CU_WEIGHT_SP, X265CU_SCALE2D_64TO32, X265CU_DEQUANT_NORMAL };
typedef struct {
    int64_t d_off, a_off, b_off;        /* element offsets into dst / srcA / srcB buffers */
    int32_t d_stride, a_stride, b_stride;
    int16_t w, h;
    int32_t p0, p1, p2, p3;             /* op parameters (shift / value / weights) */
} x265cu_blk_job;
int x265cu_blockop_batch(x265cu_ctx*, int depth, int op, void* dst_dev, const void* a_dev, const void* b_dev,
                         const x265cu_blk_job* jobs_dev, int n);

/* interpolation class (ipfilter.cpp:79-369) */
enum { X265CU_HPP = 0, X265CU_HPS, X265CU_VPP, X265CU_VPS, X265CU_VSP, X265CU_VSS, X265CU_HVPP };
typedef struct {
    int64_t s_off, d_off;
    int32_t s_stride, d_stride;
    int16_t w, h;
    int8_t  idxX, idxY, rowExt, ntaps;   /* ntaps 8 (luma) / 4 (chroma) */
} x265cu_interp_job;
int x265cu_interp_batch(x265cu_ctx*, int depth, int op, const void* src_dev, void* dst_dev,
                        const x265cu_interp_job* jobs_dev, int n);

/* transform / quant class (dct.cpp:43-742).  Blocks are n contiguous TUs. */
enum { X265CU_DCT = 0, X265CU_IDCT = 1, X265CU_DST4 = 2, X265CU_IDST4 = 3 };
/* src: strided 2-D (stride elements between rows, tu_pitch elements between TUs) for DCT;
 * dst contiguous N*N per TU.  For IDCT the roles swap (dst strided). */
int x265cu_transform_batch(x265cu_ctx*, int depth, int op, int size, const int16_t* src_dev, int16_t* dst_dev,
                           int stride, int64_t tu_pitch, int n);
/* quant over n TUs of numCoeff each; quantCoeff shared by all TUs (numCoeff entries).
 * numSig_dev[n] receives the per-TU return value.  deltaU_dev may be NULL (nquant semantics when
 * `nquant` != 0: |level| stored). */
int x265cu_quant_batch(x265cu_ctx*, const int16_t* coef_dev, const int32_t* quantCoeff_dev, int32_t* deltaU_dev,
                       int16_t* qCoef_dev, int qBits, int add, int numCoeff, int n, int nquant, uint32_t* numSig_dev);
int x265cu_dequant_normal_batch(x265cu_ctx*, const int16_t* q_dev, int16_t* coef_dev, int64_t num, int scale, int shift);
int x265cu_dequant_scaling_batch(x265cu_ctx*, const int16_t* q_dev, const int32_t* dq_dev, int16_t* coef_dev,
                                 int numCoeff, int n, int per, int shift);

/* intra class (intrapred.cpp:31-234): n jobs, each with its own 4N+1 neighbour array
 * (nb_dev + job*nb_pitch), mode, filter flag; dst block at dst_dev + job*dst_pitch, row stride dst_stride */
typedef struct { int32_t mode, bFilter; } x265cu_intra_job;
int x265cu_intra_pred_batch(x265cu_ctx*, int depth, int size, const void* nb_dev, int64_t nb_pitch,
                            void* dst_dev, int64_t dst_pitch, int dst_stride,
                            const x265cu_intra_job* jobs_dev, int n);
int x265cu_intra_filter_batch(x265cu_ctx*, int depth, int size, const void* nb_dev, void* filt_dev, int64_t pitch, int n);
int x265cu_intra_allangs_batch(x265cu_ctx*, int depth, int size, const void* ref_dev, const void* filt_dev, int64_t nb_pitch,
                               void* dst_dev, int bLuma, int n);

/* lowres (pixel.cpp:604-628 + :1027-1041): full frame -> 4 half-pel planes, margins extended */
int x265cu_frame_init_lowres(x265cu_ctx*, int depth, const void* src_dev, int src_stride,
                             void* dst0_dev, void* dsth_dev, void* dstv_dev, void* dstc_dev,
                             int dst_stride, int width, int height, int marginX, int marginY);
int x265cu_extend_border(x265cu_ctx*, int depth, void* plane_dev, int stride, int width, int height, int marginX, int marginY);

/* mvcost table (bitcost.cpp:33-110): host helper, out[2*range+1] centred */
void x265cu_mvcost_table(double lambda, int range, uint16_t* out_host);

/* motion estimation class: one job = one MotionEstimate::motionEstimate() call
 * (motion.cpp:739-1569; DIA / HEX / STAR integer search + sub-pel refine, luma).  All jobs of a
 * launch share fenc plane, stride and mvcost table; results: out_dev[job] = {cost, qmv.x, qmv.y, 0}. */
typedef struct {
    int32_t offset;             /* block origin (element offset, same in fenc and ref planes) */
    int16_t ref;                /* index into the ref plane table */
    int8_t  pw, ph;             /* PU size */
    int16_t mvmin[2], mvmax[2]; /* full-pel */
    int16_t qmvp[2];            /* qpel predictor */
    int16_t mvc[8];             /* up to 4 qpel candidates */
    int8_t  numCand, method, subme, merange;
} x265cu_me_job;
int x265cu_me_batch(x265cu_ctx*, int depth, const void* fenc_dev, int fencStride,
                    const void* const* refplanes_dev /* device array of plane ptrs */, int refStride, int lowres,
                    const uint16_t* mvcost_dev /* centred table base */, int mvcost_range,
                    const x265cu_me_job* jobs_dev, int n, int32_t* out_dev);

/* The same call with the chroma-SATD term of subpelCompare (motion.cpp:1601-1661) for 4:2:0 sources: with
 * MotionEstimate::bChromaSATD (motion.cpp:204-212: subme > 2 and PU width and height multiples of 8, so that the
 * chroma block has a SATD primitive, primitives.cpp:139-158) every sub-pel compare -- the clipped MVP, the MV
 * candidates and all refinement points -- adds SATD(Cb) + SATD(Cr) of the chroma block predicted at the eighth-pel
 * vector with the 4-tap filters.  Other jobs of the launch behave exactly as in x265cu_me_batch.
 * Chroma planes are half resolution, `cstride` pixels per row for source and references alike; the chroma pixel of the
 * luma position (x, y) = (offset % fencStride, offset / fencStride) is at (y >> 1) * cstride + (x >> 1) from the
 * pointers given.  `chroma` is a host struct of device pointers. */
typedef struct {
    const void* fencCb_dev; const void* fencCr_dev;
    const void* const* refCb_dev; const void* const* refCr_dev;   /* device arrays of plane pointers, indexed by job.ref */
    int cstride;
} x265cu_me_chroma;
int x265cu_me_batch_chroma(x265cu_ctx*, int depth, const void* fenc_dev, int fencStride,
                           const void* const* refplanes_dev, int refStride, const x265cu_me_chroma* chroma,
                           const uint16_t* mvcost_dev, int mvcost_range, const x265cu_me_job* jobs_dev, int n, int32_t* out_dev);

/* ---------- prediction costs around the motion search ----------
 * The motion-compensated prediction + cost evaluations Search::predInterSearch makes besides motionEstimate:
 *   - Search::selectMVP (encoder/search.cpp:1992-2023): SAD of the luma prediction at each AMVP candidate
 *     (predInterLumaPixel + MotionEstimate::bufSAD)                              -> cost = X265CU_PRED_SAD, one list;
 *   - Search::mergeEstimation (search.cpp:1901-1960): Predict::motionCompensation of the merge candidate (uni or bi),
 *     bufSATD + bufChromaSATD                                                     -> X265CU_PRED_SATD | X265CU_PRED_CHROMA;
 *   - the bi-directional estimate (search.cpp:2474-2607): with bChromaSATD the same motionCompensation(bi) path
 *     (addAvg of the two 14-bit intermediates, luma + chroma), without it pixelavg_pp of the two pixel predictions
 *     (luma only)                                                                -> X265CU_PRED_AVG_PP.
 * Prediction = the unweighted paths of common/predict.cpp:76-420 (4:2:0; eighth-pel chroma vector = the luma vector).
 * Vectors are quarter-pel and already clipped (CUData::clipMv, cudata.cpp:1915-1928).  The chroma term needs a chroma block
 * that is a multiple of 4x4 (motion.cpp:204-212) and chroma planes; it is skipped otherwise.  out_dev[n]: the distortion
 * (the caller adds the bit costs).  `chroma` may be NULL (no X265CU_PRED_CHROMA jobs). */
enum { X265CU_PRED_SAD = 0, X265CU_PRED_SATD = 1 };
enum { X265CU_PRED_CHROMA = 1, X265CU_PRED_AVG_PP = 2 };
typedef struct {
    int32_t offset;            /* PU origin: element offset into the luma planes (source and references share the geometry) */
    int16_t pw, ph;
    int8_t  ref0, ref1;        /* index into refplanes_dev / the chroma tables; -1 = list unused */
    uint8_t cost;              /* X265CU_PRED_SAD / X265CU_PRED_SATD */
    uint8_t flags;             /* X265CU_PRED_CHROMA | X265CU_PRED_AVG_PP */
    int16_t mv0[2], mv1[2];    /* quarter-pel */
} x265cu_pred_job;
int x265cu_pred_cost_batch(x265cu_ctx*, int depth, const void* fenc_dev, int fencStride, const void* const* refplanes_dev, int refStride,
                           const x265cu_me_chroma* chroma, const x265cu_pred_job* jobs_dev, int n, int32_t* out_dev);

/* ---------- frame-level CTU analysis (DESIGN.md "Frame analysis workload") ----------
 * One analyser = one picture geometry.  Reference planes stay resident in HBM (x265cu_analyser_set_ref
 * = what the recon-row broadcast feeds); per frame the host passes the source luma and the 16x16
 * predictor field (AMVP / lowres MVs, search.cpp:1968-2023, 2406-2410) and gets back, for every PU x
 * reference, the motionEstimate() result (motion.cpp:739), for every CU the residual-coding stats of
 * its best 2Nx2N prediction (search.cpp:3178; quant.cpp:397-470, 543-605) and its 35 intra SA8D costs
 * (search.cpp:1358-1444).  stages: bit0 ME, bit1 residual, bit2 intra. */
typedef struct x265cu_analyser x265cu_analyser;
typedef struct {
    int width, height, depth, numRefs;
    int method, subme, merange, rect;     /* X265_*_SEARCH, subpel refine level, range, rect PUs */
    int qp; double lambda;                /* quant QP; mvcost lambda (x265_lambda_tab[qp]) */
    int amp;                              /* AMP PUs (2NxnU/nD, nLx2N/nRx2N at CU >= 16; presets slower+, param.cpp:494-520) */
} x265cu_analysis_params;
typedef struct {                          /* host destinations (any may be NULL) */
    int32_t*  me_packed;                  /* [njobs][2]: cost, (mvx | mvy << 16) */
    uint64_t* cu_sse; uint32_t* cu_numsig; int32_t* cu_ref;   /* [ncu] */
    uint32_t* intra_cost;                 /* [ncu][36]: 35 costs + best mode */
} x265cu_analysis_out;
x265cu_analyser* x265cu_analyser_create(x265cu_ctx*, const x265cu_analysis_params*);
void x265cu_analyser_destroy(x265cu_analyser*);
int x265cu_analyser_counts(x265cu_analyser*, int* njobs, int* ncu, int* ntu, int64_t* ncoef, int* stride);
int x265cu_analyser_set_ref(x265cu_analyser*, int idx, const void* host_luma, int host_stride);
int x265cu_analyser_load_inputs(x265cu_analyser*, const void* fenc_host, int host_stride, const int16_t* field_host);
int x265cu_analyser_run_resident(x265cu_analyser*, int stages);       /* kernels only, inputs resident */
int x265cu_analyser_analyse(x265cu_analyser*, const void* fenc_host, int host_stride, const int16_t* field_host,
                            int stages, x265cu_analysis_out* out);    /* H2D + kernels + D2H, synchronous */
int x265cu_analyser_stage_ms(x265cu_analyser*, float ms[4]);          /* device ms of the last run: ME stage, residual, intra, ME kernel */
void* x265cu_analyser_ref_plane(x265cu_analyser*, int idx, int* stride); /* device address of ref idx's pixel (0,0) */
int x265cu_analyser_ref_updated(x265cu_analyser*, int idx);            /* re-extend borders after writing the plane in place */
int x265cu_analyser_fetch(x265cu_analyser*, int what, void* host);    /* parity/debug access to resident results */
/* CTU-row shards (BASELINE configs[4]: WPP CTU rows sharded per GPU; the reference enables row r once the reference
 * rows it needs are reconstructed, frameencoder.cpp:850-868, producer side framefilter.cpp:664).  All job / CU / TU
 * lists are in CTU raster order, so rows [ctuRow0, ctuRow1) are one contiguous slice of every result array
 * (x265cu_analyser_row_range); run_rows / analyse_rows compute exactly that slice, bit-identical to the same
 * entries of a full-frame run.  `out` arrays stay full-frame sized. */
int x265cu_analyser_ctu_rows(x265cu_analyser*);
int x265cu_analyser_row_range(x265cu_analyser*, int ctuRow0, int ctuRow1, int* job0, int* njobs, int* cu0, int* ncu);
int x265cu_analyser_run_rows(x265cu_analyser*, int stages, int ctuRow0, int ctuRow1);
int x265cu_analyser_analyse_rows(x265cu_analyser*, const void* fenc_host, int host_stride, const int16_t* field_host,
                                 int stages, int ctuRow0, int ctuRow1, x265cu_analysis_out* out);
/* 4:2:0 chroma for the chroma-SATD term of subpelCompare (MotionEstimate::bChromaSATD, motion.cpp:204-212, 1601-1661): after
 * enable_chroma() the ME stage of every run adds SATD(Cb) + SATD(Cr) to every sub-pel compare of the PUs that have a chroma
 * SATD, as the encoder does for a 4:2:0 source at subme > 2 (x265cu_me_batch_chroma's kernels on resident planes).  Upload
 * the source's chroma with load_chroma() before analyse() / run_*(), each reference's with set_ref_chroma(); host planes are
 * (width / 2) x (height / 2), host_stride in pixels. */
int x265cu_analyser_enable_chroma(x265cu_analyser*);
int x265cu_analyser_set_ref_chroma(x265cu_analyser*, int idx, const void* cb_host, const void* cr_host, int host_stride);
int x265cu_analyser_load_chroma(x265cu_analyser*, const void* cb_host, const void* cr_host, int host_stride);
void* x265cu_analyser_recon_plane(x265cu_analyser*, int depthIdx /* 0..3 = CU 64,32,16,8 */, int* stride);
int x265cu_analyser_recon_to_ref(x265cu_analyser*, int depthIdx, int refIdx, int ctuRow0, int ctuRow1);
/* Quarter-pel phase planes (X265CU_ME_PHASEPLANES, default 1; 0 = the motion search interpolates every sub-pel candidate
 * and nothing extra is allocated): every run of the ME stage first computes, per reference, the 15 fractional luma phases
 * (luma_hpp / luma_vpp / luma_hvpp) of every position its jobs can read, and the pre-checks and the sub-pel refinement read
 * their candidates from them.  Results are identical either way; the planes cost 15 extra planes of device memory per
 * reference. */
int x265cu_analyser_phase_planes_ms(x265cu_analyser*, float* ms);     /* device ms of the last run's plane build (0: none) */
void* x265cu_analyser_ref_plane_phase(x265cu_analyser*, int idx, int phase);   /* pixel (0,0) of phase (yFrac << 2) | xFrac */
int x265cu_analyser_phase_region(x265cu_analyser*, int idx, int box[4]);       /* built rectangle [x0, x1) x [y0, y1) */

/* ---------- lookahead frame costs (BASELINE configs[1]; slicetype.cpp:696-805, 3115-3388) ----------
 * All pointers are device pointers.  Planes are the 4 lowres hpel planes of a frame (origin pixel,
 * margins extended: x265cu_frame_init_lowres).  One launch handles n frames / n (p0,p1,b) triples. */
typedef struct {
    const void* plane0; const int32_t* invQscale;            /* invQscale NULL when AQ is off */
    int32_t* intraCost; uint8_t* intraMode; uint16_t* lowresCosts; int32_t* rowSatds; int64_t* out; /* out[2]: costEst, costEstAq */
} x265cu_la_intra_job;
int x265cu_lowres_intra_batch(x265cu_ctx*, int depth, const x265cu_la_intra_job* jobs_dev, int n, int stride, int w8, int h8, int lambda);
typedef struct {
    const void* fenc[4]; const void* ref0[4]; const void* ref1[4];
    int32_t* mvs[2]; int32_t* mvcosts[2];                    /* [cu][2] qpel MVs and [cu] costs per list, in/out */
    const int32_t* intraCost; const int32_t* invQscale;
    uint16_t* lowresCosts; int32_t* rowSatds; int64_t* out;  /* out[3]: costEst, costEstAq, intraMbs */
    int32_t bidir, doSearch0, doSearch1;
    int32_t rows;                                            /* 0: whole frame; else a cooperative slice (slicetype.cpp:3075-3112): CU rows [rows & 0xffff, rows >> 16) */
} x265cu_la_job;
int x265cu_lookahead_cost_batch(x265cu_ctx*, int depth, const x265cu_la_job* jobs_dev, int n, int stride, int w8, int h8,
                                const uint16_t* mvcost_dev /* centred table base, lambda of X265_LOOKAHEAD_QP */);

/* cuTree: estimateCUPropagateCost (common/pixel.cpp:914-940; EncoderPrimitives::propagateCost, primitives.h:212, 356) over
 * `len` lowres CUs -- a whole frame in one launch instead of one call per CU row (slicetype.cpp:2654-2664).  Device arrays;
 * fpsFactor as the reference passes it (slicetype.cpp:2652).  Double precision, bit-exact to the C primitive. */
int x265cu_propagate_cost_batch(x265cu_ctx*, int* dst_dev, const uint16_t* propagateIn_dev, const int32_t* intraCosts_dev,
                                const uint16_t* interCosts_dev, const int32_t* invQscales_dev, double fpsFactor, int64_t len);

/* Lookahead weighted-prediction analysis: LookaheadTLD::weightsAnalyse + weightCostLuma (slicetype.cpp:807-840, 860-961), the
 * call estimateFrameCost makes before the L0 search when --weightp is on (slicetype.cpp:3137).  Planes are whole padded
 * lowres buffers (Lowres::buffer[i], lowres.cpp:132-139: `planesize` pixels each, picture origin at `padoffset`), device
 * resident; refBuf_dev4 is a HOST array of the 4 device plane pointers; wbuf_dev (4 * planesize pixels) is
 * LookaheadTLD::wbuffer.  Host inputs: intraCost_host[CUs] (Lowres::intraCost) and stats = {fenc wp_sum, fenc wp_ssd,
 * ref wp_sum, ref wp_ssd} (Lowres::wp_sum[0] / wp_ssd[0], slicetype.cpp:49-57, 665-676).  wp_out = {isWeighted, scale,
 * log2 denominator, offset}; when isWeighted, wbuf_dev holds the 4 re-weighted planes for x265cu_lookahead_cost_batch's
 * ref0 (slicetype.cpp:3222).  The decision logic runs on the host as in the reference; the plane passes (weight_pp over
 * the padded plane, 8x8 SATD map) are launches of the block-op and grid pixel-compare kernels. */
int x265cu_lookahead_weights_analyse(x265cu_ctx*, int depth, const void* fencBuf_dev, const void* const* refBuf_dev4,
                                     void* wbuf_dev, int64_t planesize, int stride, int width, int lines, int64_t padoffset,
                                     const int32_t* intraCost_host, const uint64_t* stats, int* wp_out);

#ifdef __cplusplus
}
#endif
#endif
