/*
 * b200mvs.h — C-ABI of the B200-native dense depth estimation engine.
 *
 * Drop-in boundary for the accelerator seam of cdcseacave/openMVS:
 *   class PatchMatchCUDA { PatchMatchCUDA(int device); void Init(bool bGeomConsistency);
 *                          void Release(); void EstimateDepthMap(DepthData&); }
 *   (libs/MVS/PatchMatchCUDA.inl:78-131), owned by DepthMapsData::pmCUDA
 *   (libs/MVS/SceneDensify.h:89-92) and called from DepthMapsData::EstimateDepthMap
 *   (libs/MVS/SceneDensify.cpp:618-623), plus the SGM pair matcher
 *   SemiGlobalMatcher::Match(...) (libs/MVS/SemiGlobalMatcher.cpp:863-1302).
 *
 * Plain C: opaque context, POD structs, caller-owned buffers, int status codes
 * (0 = success; the reference exits the process on CUDA errors, libs/Common/UtilCUDA.h:81-91,
 * the adapter maps non-zero to EVT_FAIL instead).  No C++/torch types cross this boundary.
 * INTEGRATION.md shows the C++ adapter a maintainer adds on the reference side.
 */
#ifndef B200MVS_H_
#define B200MVS_H_
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200MVS_ABI_VERSION 5 /* struct layouts of this header; b200mvs_abi_version() returns the library's */
#define B200MVS_MAX_VIEWS 32 /* neighbours per reference view (MAX_VIEWS, PatchMatchCUDA.inl:35) */

typedef struct b200mvs_ctx b200mvs_ctx;

enum {
	B200MVS_OK = 0,
	B200MVS_ERR_ARG = 1,     /* invalid argument */
	B200MVS_ERR_CUDA = 2,    /* CUDA runtime error; see b200mvs_last_error() */
	B200MVS_ERR_NOGPU = 3,   /* no usable device */
	B200MVS_ERR_ALLOC = 4
};

/* One view of a DepthData (DepthData::ViewData, libs/MVS/DepthMap.h:158-185): gray float
 * image in [0,1] (Image32F from toGray(...,true), SceneDensify.cpp:324), camera K (already
 * scaled to this image size), R, C in double; optional known depth-map of the view and its
 * camera for the geometric-consistency pass (depthMap/cameraDepthMap).  views[0] is the
 * reference view. */
typedef struct {
	const float* image;   /* row-major */
	int width, height;
	int stride_bytes;     /* bytes between rows (cv::Mat::step); 0 = width*4 */
	double K[9], R[9], C[3];
	const float* depth;   /* nullable: enables the geometric term for this view */
	int dwidth, dheight, dstride_bytes;
	double Kd[9], Rd[9], Cd[3];
	/* Alternative to `image` (used when image == NULL): the 8-bit colour image as cv::imread delivers it, converted on the
	 * device with the reference's toGray(..., bNormalize = true) arithmetic (libs/Common/Types.inl:2377-2431, applied by
	 * InitViews, SceneDensify.cpp:324,345).  The host path then uploads 3 bytes per pixel instead of 4. */
	const uint8_t* image8; /* width x height x channels8, row-major */
	int channels8;         /* 3 or 4 interleaved channels */
	int bgr8;              /* != 0: B,G,R order (cv::imread); 0: R,G,B */
	int stride8_bytes;     /* bytes between rows; 0 = width*channels8 */
} b200mvs_view;

/* Snapshot of the OPTDENSE knobs the estimator consumes (libs/MVS/DepthMap.cpp:69-114),
 * taken at call time because the reference mutates some of them during a run
 * (fNCCThresholdKeep, SceneDensify.cpp:775-796). */
typedef struct {
	int nEstimationIters;                   /* 3  */
	int nEstimationGeometricIters;          /* 2  */
	int nRandomIters;                       /* 6  */
	int nSubResolutionLevels;               /* 2  */
	float fNCCThresholdKeep;                /* 0.9 */
	float fDescriptorMinMagnitudeThreshold; /* 0.02 */
	float fRandomDepthRatio;                /* 0.003 */
	float fRandomAngle1Range;               /* 16 (deg) */
	float fRandomAngle2Range;               /* 10 (deg) */
	float fRandomSmoothDepth;               /* 0.02 */
	float fRandomSmoothNormal;              /* 13 (deg) */
	float fRandomSmoothBonus;               /* 0.93 */
	float fEstimationGeometricWeight;       /* 0.1 */
	/* engine schedule (not OPTDENSE; DESIGN.md §2).  The nEstimationIters reference iterations run as red-black sweeps:
	 * nSweepsPerIter = 0 (default): max(8, ceil(1.5 x nEstimationIters)) sweeps that share the reference's
	 * nRandomIters x nEstimationIters refinement tries; > 0: nSweepsPerIter sweeps per iteration, each with
	 * ceil(nRandomIters/nSweepsPerIter) tries.  b200mvs_get_schedule() returns the resulting numbers. */
	int nSweepsPerIter;                     /* 0  */
	int nPropagation;                       /* 4: all 4-neighbours; 2: causal pair only */
	uint32_t seed;                          /* Philox key */
	int nPropagationFar;                    /* 2: per direction the candidate is the lowest-cost pixel at distance 1, 3, .. 2n+1 (0: adjacent only) */
	int bSkipUnchanged;                     /* 1: a direction whose candidates kept their plane in their last update is not re-tested */
	int nEvalCap;                           /* 7: a pixel that tests c propagation candidates in a sweep spends at most max(1, nEvalCap - c)
	                                           refinement tries in it (0: always nRandomIters-derived tries) */
} b200mvs_params;

/* Diagnostic switches (all zero = the shipped kernels); replaces the environment variables of round 1. */
typedef struct {
	int scalarTaps;      /* 1: bilinear taps one at a time instead of the packed FMUL2/FFMA2 form (bit-identical results) */
	int noTMA;           /* 1: the sweep kernel reads the reference patch with plain loads instead of the TMA-staged tile */
	int sgmAggregation;  /* 0 auto; 1 general ragged kernel; 2 register-pipelined uniform kernel; 3 bulk-copy ring kernel (one launch
	                        per direction); 4 front kernel (fused directions, auto default for uniform ranges) */
	int sgmCost;         /* 0 auto (tensor-core kernel for dense volumes with one range of 64 / 128 / 192 / 256 disparities, SIMT otherwise);
	                        1 SIMT cost kernel; 2 tensor-core (tcgen05) cost kernel or an error */
	int sweepFourCtas;   /* 1: the 64-register instantiation of the sweep kernel (4 CTAs per SM instead of 3) */
	int frontLayout;     /* wave-front aggregation: 0 auto; 1 two tilted fronts +-(x+2y), four directions each; 2 four straight
	                        fronts; 3 eight passes of one direction */
	int frontSerial;     /* 1: one pass per launch into one sum volume (default: two passes share a launch, each with its own
	                        volume, added by the winner-takes-all kernel) */
	int frontBlock;      /* fronts per work item (0: default) */
	int frontLag;        /* 1 + queue distance, in blocks, between the directions of a pass (0: default = distance 1) */
	int frontCtas;       /* resident CTAs per SM (0: default) */
	int frontDepth;      /* steps whose loads are in flight: 4 or 8 (0: default) */
	int frontSubCell;    /* columns per sub-cell of the phase dependencies (0: default 64; never fewer than width / 30) */
	int reserved[4];
} b200mvs_debug;

typedef struct {
	double ms_total;      /* wall time of the call (host clock) */
	double ms_device;     /* device time between first and last kernel (CUDA events) */
	uint64_t bytes_h2d, bytes_d2h;
	int kernel_launches;
	int levels;
	double ms_sweep_kernels; /* summed device time of the red-black half-sweep launches (CUDA events) */
	int sweep_launches;
	int tma_active;          /* 1: the sweep kernels staged the reference tile with TMA (cp.async.bulk.tensor) */
} b200mvs_stats;

/* ---- lifetime (PatchMatchCUDA ctor / Init / Release, PatchMatchCUDA.cpp:60-117) ---- */
int  b200mvs_create(int device, b200mvs_ctx** ctx);
int  b200mvs_destroy(b200mvs_ctx* ctx);
void b200mvs_default_params(b200mvs_params* p);
int  b200mvs_set_params(b200mvs_ctx* ctx, const b200mvs_params* p);
int  b200mvs_set_debug(b200mvs_ctx* ctx, const b200mvs_debug* d /* NULL: defaults */);
/* sweeps and refinement tries per sweep the engine runs for p (geometric != 0: for one geometric-consistency pass) */
int  b200mvs_get_schedule(const b200mvs_params* p, int geometric, int* nSweeps, int* nRefinePerSweep);
int  b200mvs_abi_version(void);
size_t b200mvs_sizeof(int what); /* 0 view, 1 params, 2 stats, 3 job, 4 sgm_pixel, 5 sgm_params, 6 dmap, 7 filter_params, 8 debug */
/* Ignore-mask of the reference view for the following estimate calls (OPTDENSE::nIgnoreMaskLabel >= 0:
 * DepthEstimator::ImportIgnoreMask + DepthData::ApplyIgnoreMask, libs/MVS/DepthMap.cpp:215-230,300-323;
 * SceneDensify.cpp:660-664,679-693): one byte per pixel of the full-resolution reference image, 0 = ignored.  Ignored pixels
 * are neither scored nor swept (depth = normal = conf = 0), every pyramid level uses the NEAREST-resized mask and the depth is
 * up-sampled NEAREST instead of LINEAR, like the CPU path.  mask = NULL clears it.  on_device != 0: `mask` is a device pointer
 * that stays valid until cleared; otherwise the host buffer is copied during the call. */
int  b200mvs_set_ignore_mask(b200mvs_ctx* ctx, const uint8_t* mask, int width, int height, int stride_bytes, int on_device);
const char* b200mvs_last_error(const b200mvs_ctx* ctx);
int  b200mvs_device_count(void);

/* ---- DepthMapsData::EstimateDepthMap(idxImage, nGeometricIter) replacement ------------
 * (SceneDensify.cpp:616-805 / PatchMatchCUDA::EstimateDepthMap, PatchMatchCUDA.cpp:174-416)
 * HOST buffers.  depth/normal are in/out (initial estimate; depth outside [dMin,dMax) =>
 * random init), conf and viewsMap out.  nGeometricIter < 0: photometric pass with the
 * scale loop; >= 0: one geometric-consistency iteration (views[i].depth required).
 * Output follows EndDepthMapTmp: rejected pixels have depth=0, normal=0, conf=0; others
 * conf = 1-cost.  viewsMap (nullable): 4 x uint8 per pixel, the neighbour indices that
 * produced the score, 255 padding (PatchMatchCUDA.cpp:374-391). */
int b200mvs_estimate(b200mvs_ctx* ctx, const b200mvs_view* views, int nViews,
	float dMin, float dMax, int nGeometricIter,
	float* depth, float* normal, float* conf, uint8_t* viewsMap, b200mvs_stats* stats);

/* Asynchronous form of b200mvs_estimate: enqueues the H2D copies, the kernels and the D2H copies on the
 * context's stream and returns; host buffers (pinned for real overlap) must stay valid until
 * b200mvs_sync(ctx, stats) returns.  Two contexts used alternately overlap the copies of one reference view
 * with the kernels of the other — what the reference's two worker threads do around the seam
 * (SceneDensify.cpp:1893-1899, 2036-2059). */
int b200mvs_estimate_async(b200mvs_ctx* ctx, const b200mvs_view* views, int nViews,
	float dMin, float dMax, int nGeometricIter,
	float* depth, float* normal, float* conf, uint8_t* viewsMap);
int b200mvs_sync(b200mvs_ctx* ctx, b200mvs_stats* stats);

/* One reference-view job of a batch: the arguments of b200mvs_estimate */
typedef struct {
	const b200mvs_view* views; int nViews;
	float dMin, dMax; int nGeometricIter;
	float* depth; float* normal; float* conf; uint8_t* viewsMap;
	int status;            /* out: status code of this job */
} b200mvs_job;

/* Batch form for per-reference-view parallelism inside ONE process: jobs are dealt round-robin over the
 * given contexts (one per GPU of the box, or two on one GPU for copy/compute overlap) through
 * b200mvs_estimate_async, each context is drained with b200mvs_sync before it is reused.  Reference views
 * are independent (SceneDensify.cpp:2036-2059 estimates them one by one), so there is no data-path
 * collective.  Returns the first non-zero job status (all jobs are attempted). */
int b200mvs_estimate_batch(b200mvs_ctx** ctxs, int nCtx, b200mvs_job* jobs, int nJobs);

/* Same, but every pointer inside `views` and the map pointers are DEVICE pointers on the
 * context's device (data resident in HBM); work is enqueued on `stream` (cudaStream_t; NULL = the
 * context's own non-blocking stream, pass cudaStreamLegacy for the legacy default stream) and
 * the call returns after enqueueing unless stats != NULL (then it synchronises). */
int b200mvs_estimate_device(b200mvs_ctx* ctx, const b200mvs_view* views, int nViews,
	float dMin, float dMax, int nGeometricIter,
	float* depth, float* normal, float* conf, uint8_t* viewsMap, void* stream, b200mvs_stats* stats);

/* ---- building blocks (device pointers), exposed for parity tests ----------------------
 * state: plane = float4 {nx,ny,nz,depth} per pixel, cost = raw score in [0,2]. */
int b200mvs_pm_pack(b200mvs_ctx* ctx, int width, int height, const float* depth, const float* normal,
	float* plane4, void* stream);
int b200mvs_pm_unpack(b200mvs_ctx* ctx, int width, int height, const float* plane4,
	float* depth, float* normal, void* stream);
/* pass A — ScoreDepthMapTmp (SceneDensify.cpp:490-517) */
int b200mvs_pm_score(b200mvs_ctx* ctx, const b200mvs_view* views, int nViews, float dMin, float dMax,
	const float* lowres, float* plane4, float* cost, void* stream);
/* pass B — one red-black sweep `sweep` (EstimateDepthMapTmp/ProcessPixel); half = -1 both
 * colours, 0/1 a single colour */
int b200mvs_pm_sweep(b200mvs_ctx* ctx, const b200mvs_view* views, int nViews, float dMin, float dMax,
	const float* lowres, int sweep, int half, int nRandomIters, float* plane4, float* cost, void* stream);
/* pass C — EndDepthMapTmp (SceneDensify.cpp:528-548) */
int b200mvs_pm_finalize(b200mvs_ctx* ctx, int width, int height, float keepThreshold,
	const float* plane4, const float* cost, float* depth, float* normal, float* conf, void* stream);

/* ---- SemiGlobalMatcher::Match(leftImage, rightImage, disparityMap, costMap) replacement -------
 * (libs/MVS/SemiGlobalMatcher.cpp:863-1302; WZNCC 7x7 cost, 8-path aggregation with per-pixel
 * disparity ranges, winner-takes-all).  Images are rectified: left/right gray float (sRGB->linear,
 * SemiGlobalMatcher.cpp:580-581) and the left colour image (BGR, 3 x uint8), all width x height.
 * `pixels` is the reference's PixelMap over the valid region (width-6) x (height-6):
 * idx = offset of the pixel's first cost in the ragged volume, [dmin,dmax) its disparity range
 * (dmin >= dmax: invalid pixel, skipped; PixelData, SemiGlobalMatcher.h:78-81).  numCosts = total
 * number of (pixel, disparity) entries.  Outputs over the valid region: disparity (int16) and the
 * summed path cost (uint16, 65535 for invalid pixels). */
typedef struct {
	uint64_t idx;
	int16_t dmin, dmax;
	int32_t reserved;
} b200mvs_sgm_pixel;

typedef struct {
	int P1;            /* 3  (SemiGlobalMatcher ctor defaults, SemiGlobalMatcher.h:149) */
	int P2;            /* 4  */
	float P2alpha;     /* 14 */
	float P2beta;      /* 38 */
} b200mvs_sgm_params;

void b200mvs_sgm_default_params(b200mvs_sgm_params* p);

/* HOST buffers */
int b200mvs_sgm_match(b200mvs_ctx* ctx, const float* leftGray, const uint8_t* leftBGR, const float* rightGray,
	int width, int height, const b200mvs_sgm_pixel* pixels, uint64_t numCosts, const b200mvs_sgm_params* prm,
	int16_t* disparity, uint16_t* cost, b200mvs_stats* stats);

/* DEVICE pointers.  stages: bit 0 compute the cost volume, bit 1 aggregate the 8 paths, bit 2
 * winner-takes-all.  costs (uint8) / accums (uint16) hold numCosts entries; pass NULL to use the
 * context's scratch, or buffers to inspect / supply the volumes (parity tests feed the oracle's cost
 * volume into the aggregation). */
int b200mvs_sgm_match_device(b200mvs_ctx* ctx, const float* leftGray, const uint8_t* leftBGR, const float* rightGray,
	int width, int height, const b200mvs_sgm_pixel* pixels, uint64_t numCosts, const b200mvs_sgm_params* prm,
	int stages, uint8_t* costs, uint16_t* accums, int16_t* disparity, uint16_t* cost, void* stream, b200mvs_stats* stats);

/* ConsistencyCrossCheck(l2r, r2l, thCross) (SemiGlobalMatcher.cpp:1449-1489), DEVICE pointers, l2r in place:
 * a left disparity survives if the right disparity it points to is valid and |ld + rd| <= thCross. */
int b200mvs_sgm_cross_check_device(b200mvs_ctx* ctx, int16_t* l2r, const int16_t* r2l, int width, int height,
	int thCross, void* stream);

/* RefineDisparityMap (SemiGlobalMatcher.cpp:1693-1811) with SUBPIXEL_LC_BLEND: sub-pixel offset from the
 * accumulated costs around the winner, result stored as round(disparity * subpixelSteps).  DEVICE pointers;
 * accums = NULL uses the accumulated costs of the last match on this context. */
int b200mvs_sgm_refine_device(b200mvs_ctx* ctx, const b200mvs_sgm_pixel* pixels, const uint16_t* accums,
	int16_t* disparity, int nPixels, int subpixelSteps, void* stream);

/* ---- coarse-to-fine (tSGM) matching of a rectified pair: the level loop of SemiGlobalMatcher::Match(scene, idxImage, numNeighbors,
 * minResolution) (libs/MVS/SemiGlobalMatcher.cpp:584-718), the reference's default SGM path, between StereoRectifyImages and
 * ExportDisparityDataRawFull.  Levels at 1/2^L .. 1/2, 1 of the full resolution: the coarsest level matches inside ranges derived
 * from a seed disparity map, every finer level inside per-pixel ranges of at most 64 disparities derived from the level below, so
 * the total disparity span is not limited to 256.
 * b200mvs_sgm_tsgm_levels: number of levels (computeMaxResolution, libs/Common/Types.inl:2459-2477, minResolution > 0) and the size of
 * the seed: computeResize(coarsest level, 0.5) minus 6 in each dimension (234 x 129 for 1920 x 1080). */
int b200mvs_sgm_tsgm_levels(int width, int height, int minResolution, int* nLevels, int* seedWidth, int* seedHeight);

/* DEVICE pointers, work on `stream` (NULL = the context's stream).  Images as b200mvs_sgm_match plus the right BGR image; masks
 * (nullable = all valid): width x height bytes, 0 = invalid (StereoRectifyImages); maskWidth / maskHeight must equal width / height
 * when a mask is given.  seed (nullable = all unknown): seedWidth x seedHeight int16 disparities at half the coarsest scale,
 * 32767 = unknown.  nSpeckleSize: OPTDENSE::nSpeckleSize (100); subpixelSteps: 4; prm NULL = defaults.  Outputs over the
 * (width-6) x (height-6) valid region: the refined left disparity x subpixelSteps (32767 = none) and the cost of the last left match.
 * Synchronises the stream once per match (two per level), where the ragged cost volume is sized from the pixel map; when a match
 * took the wave-front aggregation, once more to read its timeout flag.  stats != NULL: also at the end.  Scratch is grow-only on
 * the context.  B200MVS_ERR_ARG for wrong seed or mask sizes, or an image too small for minResolution. */
int b200mvs_sgm_match_tsgm_device(b200mvs_ctx* ctx, const float* leftGray, const uint8_t* leftBGR, const float* rightGray, const uint8_t* rightBGR,
	int width, int height, const uint8_t* leftMask, const uint8_t* rightMask, int maskWidth, int maskHeight,
	const int16_t* seed, int seedWidth, int seedHeight, int minResolution, int nSpeckleSize, int subpixelSteps,
	const b200mvs_sgm_params* prm, int16_t* disparity, uint16_t* cost, void* stream, b200mvs_stats* stats);
/* Same with HOST buffers: copies in, runs the device form on the context's stream, copies out. */
int b200mvs_sgm_match_tsgm(b200mvs_ctx* ctx, const float* leftGray, const uint8_t* leftBGR, const float* rightGray, const uint8_t* rightBGR,
	int width, int height, const uint8_t* leftMask, const uint8_t* rightMask, int maskWidth, int maskHeight,
	const int16_t* seed, int seedWidth, int seedHeight, int minResolution, int nSpeckleSize, int subpixelSteps,
	const b200mvs_sgm_params* prm, int16_t* disparity, uint16_t* cost, b200mvs_stats* stats);

/* building blocks of the level loop (DEVICE pointers) */
/* Disparity2RangeMap (SemiGlobalMatcher.cpp:1350-1444): ranges at twice the scale of `disparity` (width x height) over the finer
 * valid region `mask` (maskWidth >= 2 width + 4, maskHeight >= 2 height + 2); pixels receives maskWidth x maskHeight records.
 * Synchronises `stream` to return *numCosts and *maxNumDisp (nullable). */
int b200mvs_sgm_range_map_device(b200mvs_ctx* ctx, const int16_t* disparity, int width, int height, const uint8_t* mask, int maskWidth, int maskHeight,
	int minNumDisp, int minNumDispInvalid, b200mvs_sgm_pixel* pixels, uint64_t* numCosts, int* maxNumDisp, void* stream);
/* FlipDirection (SemiGlobalMatcher.cpp:1630-1657): r2l = NO_DISP, every valid l2r(r,c) = d writes -d to r2l(r, c+d-1 .. c+d+1);
 * where writes overlap the larger source column wins */
int b200mvs_sgm_flip_direction_device(b200mvs_ctx* ctx, const int16_t* l2r, int16_t* r2l, int width, int height, void* stream);
/* cv::filterSpeckles(disparity, newVal, maxSpeckleSize, maxDiff) on int16, in place */
int b200mvs_sgm_filter_speckles_device(b200mvs_ctx* ctx, int16_t* disparity, int width, int height, int newVal, int maxSpeckleSize, int maxDiff, void* stream);
/* ExtractMask (SemiGlobalMatcher.cpp:1518-1575): mask (same size) updated in place */
int b200mvs_sgm_extract_mask_device(b200mvs_ctx* ctx, const int16_t* disparity, uint8_t* mask, int width, int height, int thValid, void* stream);
/* UpscaleMask (SemiGlobalMatcher.cpp:1662-1690) into mask2x (width2 x height2) */
int b200mvs_sgm_upscale_mask_device(b200mvs_ctx* ctx, const uint8_t* mask, int width, int height, uint8_t* mask2x, int width2, int height2, void* stream);
/* cv::resize(image, Size(), 1./factor, 1./factor, INTER_AREA) of a 3-channel 8-bit image (integer factor >= 2); `resized` holds
 * cvRound(width/factor) x cvRound(height/factor) pixels */
int b200mvs_resize_area_bgr8_device(b200mvs_ctx* ctx, const uint8_t* image, int width, int height, int factor, uint8_t* resized, void* stream);

/* ---- depth-map post-processing after the estimation (SURVEY.md §8(f) rank 2) -----------------
 * DepthMapsData::FilterDepthMap / RemoveSmallSegments / GapInterpolation
 * (libs/MVS/SceneDensify.cpp:1050-1299, 810-900, 904-1045).  Maps are contiguous row-major float
 * (cv::Mat-backed DepthMap / ConfidenceMap / NormalMap).  The OPTDENSE values are passed raw; the
 * per-function multipliers (x1.2 / x0.8, x0.7, x2.5) are applied inside, as in the reference. */
#define B200MVS_MAX_FILTER_VIEWS 16 /* the reference uses at most numMaxNeighbors = 8 (SceneDensify.cpp:2152) */

/* an estimated depth-map with the camera it was estimated in (DepthData: depthMap, confMap,
 * images.First().camera) */
typedef struct {
	const float* depth;   /* width x height */
	const float* conf;    /* width x height; may be NULL for neighbours when bAdjust = 0 */
	int width, height;
	double K[9], R[9], C[3];
} b200mvs_dmap;

typedef struct {
	int nMinViews;              /* min(OPTDENSE::nMinViewsFilter = 2, nCalibratedImages-1) */
	int nMinViewsAdjust;        /* min(OPTDENSE::nMinViewsFilterAdjust = 1, nCalibratedImages-1) */
	float fDepthDiffThreshold;  /* OPTDENSE::fDepthDiffThreshold = 0.01 */
	int bAdjust;                /* OPTDENSE::bFilterAdjust = 1 */
} b200mvs_filter_params;

void b200mvs_filter_default_params(b200mvs_filter_params* p);

/* FilterDepthMap(depthDataRef, idxNeighbors, bAdjust): z-buffered projection of the nNbrs neighbour
 * depth-maps into the reference view, then per pixel either the confidence-weighted average of the
 * agreeing depths (bAdjust) or a keep/discard vote.  HOST buffers; outDepth/outConf are the
 * "filtered.dmap"/"filtered.cmap" maps the reference saves.  *filtered (nullable) receives 0 when the
 * map can not be filtered (nNbrs < nMinViews or < nMinViewsAdjust; outputs untouched), else 1. */
int b200mvs_filter_depth_map(b200mvs_ctx* ctx, const b200mvs_dmap* ref, const b200mvs_dmap* nbrs, int nNbrs,
	const b200mvs_filter_params* prm, float dMin, float dMax, float* outDepth, float* outConf, int* filtered,
	b200mvs_stats* stats);
/* Same with DEVICE pointers inside ref/nbrs and for the outputs (outputs must not alias the inputs).
 * projDepth / projConf (nullable, nNbrs x height x width) receive the projected neighbour maps. */
int b200mvs_filter_depth_map_device(b200mvs_ctx* ctx, const b200mvs_dmap* ref, const b200mvs_dmap* nbrs, int nNbrs,
	const b200mvs_filter_params* prm, float dMin, float dMax, float* outDepth, float* outConf,
	float* projDepth, float* projConf, int* filtered, void* stream);

/* RemoveSmallSegments(depthData): zero every 4-connected segment of similar depths
 * (threshold fDepthDiffThreshold*0.7) smaller than nSpeckleSize pixels; in place; normal / conf nullable.
 * Segments are the reference's: grown breadth-first from seeds in column-major order with the directed test
 * IsDepthSimilar(current, neighbour) (SceneDensify.cpp:828-895).  The device form reads the (few) one-way edges back to
 * resolve them on the host, so it synchronises `stream` once. */
int b200mvs_remove_small_segments(b200mvs_ctx* ctx, float* depth, float* normal, float* conf, int width, int height,
	float fDepthDiffThreshold, unsigned nSpeckleSize, b200mvs_stats* stats);
int b200mvs_remove_small_segments_device(b200mvs_ctx* ctx, float* depth, float* normal, float* conf, int width, int height,
	float fDepthDiffThreshold, unsigned nSpeckleSize, void* stream);

/* GapInterpolation(depthData): fill row gaps, then column gaps, of at most nIpolGapSize invalid pixels
 * between two similar depths (threshold fDepthDiffThreshold*2.5) by linear interpolation of the depth and
 * of the normal's direction angles; confidence = min of the two ends; in place; normal / conf nullable. */
int b200mvs_gap_interpolation(b200mvs_ctx* ctx, float* depth, float* normal, float* conf, int width, int height,
	float fDepthDiffThreshold, unsigned nIpolGapSize, b200mvs_stats* stats);
int b200mvs_gap_interpolation_device(b200mvs_ctx* ctx, float* depth, float* normal, float* conf, int width, int height,
	float fDepthDiffThreshold, unsigned nIpolGapSize, void* stream);

/* ---- image preparation before the estimation (SURVEY.md §8(f) rank 3) -------------------------
 * TImage<Pixel8U>::toGray(out, cv::COLOR_BGR2GRAY, bNormalize = true) (libs/Common/Types.inl:2377-2431), applied by
 * DepthMapsData::InitViews to every image (SceneDensify.cpp:324,345): 8-bit colour image (3 or 4 interleaved channels,
 * bgr != 0: B,G,R order as cv::imread delivers; 0: R,G,B) -> float gray in [0,1], coefficients .114 / .587 / .299.
 * DEVICE pointers: upload the 8-bit image once (3 B per pixel instead of 4) and convert in HBM; strides in bytes, 0 = packed. */
int b200mvs_to_gray_device(b200mvs_ctx* ctx, const uint8_t* image, int width, int height, int stride_bytes, int channels, int bgr,
	float* gray, int gray_stride_bytes, void* stream);

/* DepthData::ViewData::ScaleImage (libs/MVS/DepthMap.h:193-203), applied by DepthMapsData::InitViews to a neighbour whose footprint
 * scale differs from 1 by 15 % or more (SceneDensify.cpp:324-326,345-347): cv::resize(image, Size(), scale, scale,
 * scale > 1 ? INTER_CUBIC : INTER_AREA) of the float gray image; the caller recomputes the camera for the new size
 * (Image::GetCamera).  b200mvs_scaled_size gives the size cv::resize produces.  DEVICE pointers; `scaled` holds
 * scaledWidth x scaledHeight contiguous floats.  *applied (nullable) = 0 when |scale - 1| < 0.15 (nothing written), else 1. */
int b200mvs_scaled_size(int width, int height, float scale, int* scaledWidth, int* scaledHeight);
int b200mvs_scale_image_device(b200mvs_ctx* ctx, const float* image, int width, int height, int stride_bytes, float scale,
	float* scaled, int* applied, void* stream);

/* ---- fusion of the depth-maps into a point cloud (SURVEY.md §8(f) rank 4) -----------------------
 * DepthMapsData::FuseDepthMaps (libs/MVS/SceneDensify.cpp:1372-1646): HOST arrays, host code — the result depends on the order in
 * which points claim pixels and zero blocking depths, so the reference's sequential loop is the specification (best connected
 * images first, pixels in raster order).  One b200mvs_fuse_view per scene image (index = image ID); images without a depth-map
 * have depth = NULL.  `depth` is modified like the reference modifies its depth-maps (depths behind an accepted point become 0). */
typedef struct {
	int width, height;            /* size of the maps (and of `color`) */
	float* depth;                 /* in/out; NULL: no depth-map */
	const float* normal;          /* camera-space unit normals, 3 floats per pixel, or NULL */
	const float* conf;            /* confidence in [0,1] or NULL (weight 1) */
	const uint8_t* color;         /* 3 bytes per pixel (the image at map resolution) or NULL */
	double K[9], R[9], C[3];      /* camera at map resolution */
	const uint32_t* neighbors;    /* depthData.neighbors: image IDs, best first */
	int nNeighbors;
	int nSceneNeighbors;          /* scene.images[i].neighbors.size(): the connection score (images are fused best connected first) */
} b200mvs_fuse_view;
typedef struct {
	int nMinViewsFuse;            /* 2 (OPTDENSE::nMinViewsFuse, libs/MVS/DepthMap.cpp:75) */
	float fDepthDiffThreshold;    /* 0.01 */
	float fNormalDiffThreshold;   /* 25 (degrees) */
	int bEstimateColor;           /* 1 */
	int bEstimateNormal;          /* 1 */
} b200mvs_fuse_params;
typedef struct b200mvs_pointcloud b200mvs_pointcloud;   /* PointCloud: points, pointViews, pointWeights, colors, normals */
void b200mvs_fuse_default_params(b200mvs_fuse_params* p);
int b200mvs_fuse_depth_maps(b200mvs_fuse_view* views, int nViews, const b200mvs_fuse_params* prm, b200mvs_pointcloud** cloud);
uint64_t b200mvs_pointcloud_size(const b200mvs_pointcloud* cloud);
uint64_t b200mvs_pointcloud_depths(const b200mvs_pointcloud* cloud);               /* valid depths visited (the reference's nDepths) */
const float* b200mvs_pointcloud_points(const b200mvs_pointcloud* cloud);           /* 3 floats per point */
const float* b200mvs_pointcloud_normals(const b200mvs_pointcloud* cloud);          /* 3 floats per point or NULL */
const uint8_t* b200mvs_pointcloud_colors(const b200mvs_pointcloud* cloud);         /* 3 bytes per point or NULL */
const uint32_t* b200mvs_pointcloud_view_offsets(const b200mvs_pointcloud* cloud);  /* size+1 entries: views / weights of point i are [o[i], o[i+1]) */
const uint32_t* b200mvs_pointcloud_views(const b200mvs_pointcloud* cloud);         /* image IDs, ascending per point */
const float* b200mvs_pointcloud_weights(const b200mvs_pointcloud* cloud);
const uint16_t* b200mvs_pointcloud_projs(const b200mvs_pointcloud* cloud);         /* pixel (x, y) of every view of every point */
void b200mvs_pointcloud_free(b200mvs_pointcloud* cloud);

#ifdef __cplusplus
}
#endif
#endif /* B200MVS_H_ */
