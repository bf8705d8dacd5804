// capi.cu — host side of the C-ABI declared in include/b200mvs.h.
//
// Mirrors the control flow of DepthMapsData::EstimateDepthMap (libs/MVS/SceneDensify.cpp:616-805)
// and of the accelerator seam PatchMatchCUDA::EstimateDepthMap (libs/MVS/PatchMatchCUDA.cpp:174-416):
// scale loop -> pass A (score) -> pass B (sweeps) -> pass C (threshold), all on one stream,
// no host synchronisation between kernels.
#include "../../include/b200mvs.h"
#include "pm_common.cuh"
#include "sgm_front_sched.h"
#include <cuda.h>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>
#include <chrono>
#include <algorithm>
#include <cstdlib>

cudaError_t pm_configure_device();
cudaError_t pm_launch_score(const PMParams& P, bool pack, bool geom, cudaStream_t s);
cudaError_t pm_launch_sweep(const PMParams& P, const void* tmapRef, bool pack, bool geom, bool fourCtas, cudaStream_t s);
void pm_tma_box(int* w, int* h);
cudaError_t pm_launch_finalize(int n, float keep, const float4* plane, const float* cost, const uint32_t* bestViews,
	float* depth, float* normal, float* conf, uint32_t* viewsMap, cudaStream_t s);
cudaError_t pm_launch_pack(int n, const float* depth, const float* normal, float4* plane, cudaStream_t s);
cudaError_t pm_launch_unpack(int n, const float4* plane, float* depth, float* normal, cudaStream_t s);
struct SGMPixel { unsigned long long idx; short dmin, dmax; int pad; };
struct SGMParams {
	const float* lgray; const uchar3* lbgr; const float* rgray;
	int w, h, vw, vh;
	const SGMPixel* px;
	uint8_t* costs; uint16_t* accums;
	int P1;
	uint16_t P2s[256];
	int maxNumDisp;
};
cudaError_t sgm_configure_device();
cudaError_t sgm_launch_maxdisp(const SGMPixel* px, int n, unsigned long long numCosts, int* out8, cudaStream_t s);
cudaError_t sgm_launch_cost(const SGMParams& P, cudaStream_t s);
cudaError_t sgm_cost_tc_configure();
bool sgm_cost_tc_supports(int num);
cudaError_t sgm_cost_tc_launch(const SGMParams& P, int dmin, int num, cudaStream_t s);
cudaError_t sgm_launch_aggregate(const SGMParams& P, int dir, bool store, cudaStream_t s);
cudaError_t sgm_launch_aggregate_uniform(const SGMParams& P, int dir, int dmin, int num, bool ring, cudaStream_t s);
// wave-front aggregation (sgm_front.cu)
cudaError_t sgm_front_launch(const SGMParams& P, const FrontArgs& A, int blocks, int pd, cudaStream_t s);
int sgm_front_blocks_per_sm(int num, int pd);
bool sgm_front_supports(int num);
cudaError_t sgm_launch_wta(const SGMParams& P, int nVol, unsigned long long volStride, const uint16_t* more, int16_t* disparity, uint16_t* cost, cudaStream_t s);
cudaError_t sgm_launch_wta_uniform(const SGMParams& P, const uint16_t* second, int dmin, int num, int16_t* disparity, uint16_t* cost, cudaStream_t s);
int sgm_max_disparities();
cudaError_t sgm_launch_cross_check(int16_t* l2r, const int16_t* r2l, int w, int h, int th, cudaStream_t s);
cudaError_t sgm_launch_refine(const SGMPixel* px, const uint16_t* accums, int16_t* disparity, int n, int steps, cudaStream_t s);
#define FLT_MAX_NBR 16
struct FltView { const float* depth; const float* conf; int w, h; double fx, fy, cx, cy; double R[9], C[3]; };
struct FltParams {
	FltView ref; FltView nbr[FLT_MAX_NBR];
	int N, nMinViews, nMinViewsAdjust;
	float thDepthDiff, thStrict, dMin, dMax;
	unsigned long long* zbuf; float* outDepth; float* outConf;
};
cudaError_t flt_launch_filter(const FltParams& P, int maxNbrPixels, bool adjust, cudaStream_t s);
cudaError_t flt_launch_resolve(const unsigned long long* z, const float* nbrConf, size_t np, float* depth, float* conf, cudaStream_t s);
struct SegArc { int src, dst, srcSize, dstSize, srcKey, dstKey; };
cudaError_t seg_launch_label(const float* depth, int W, int H, float th, int* labels, int* sizes, int* minKey, void* arcs, int* count, int cap, cudaStream_t s);
cudaError_t seg_launch_remove(float* depth, float* normal, float* conf, int W, int H, unsigned speckle, const int* labels, int* sizes,
	const int* patch, int nPatch, cudaStream_t s);
cudaError_t gap_launch(float* depth, float* normal, float* conf, float* tDepth, float* tNormal, float* tConf, int W, int H, float th, int gap, cudaStream_t s);
cudaError_t rs_launch_area(const float* src, int sw, int sh, int spitch, float* dst, int dw, int dh, double scx, double scy, cudaStream_t s);
cudaError_t rs_launch_cubic(const float* src, int sw, int sh, int spitch, float* dst, int dw, int dh, int dpitch, double scx, double scy, cudaStream_t s);
cudaError_t rs_launch_linear(const float* src, int sw, int sh, float* dst, int dw, int dh, cudaStream_t s);
cudaError_t rs_launch_nearest(const float* src, int sw, int sh, int ch, float* dst, int dw, int dh, double scx, double scy, cudaStream_t s);
cudaError_t rs_launch_nearest_u8(const uint8_t* src, int sw, int sh, int spitch, uint8_t* dst, int dw, int dh, cudaStream_t s);
cudaError_t rs_launch_to_gray(const uint8_t* src, int w, int h, int sstride, int channels, int bgr, float* dst, int dpitch, cudaStream_t s);
cudaError_t rs_launch_plane_up(const float4* src, int sw, int sh, float4* dst, float* prior, int dw, int dh, bool nearestDepth, cudaStream_t s);
// coarse-to-fine SGM steps (sgm_tsgm.cu)
size_t ts_range_scratch_bytes(int mw, int mh);
cudaError_t ts_launch_range_map(const int16_t* D, int dw, int dh, const uint8_t* M, int mw, int mh, int minNumDisp, int minNumDispInvalid,
	uint32_t* range, void* scratch, void* pixels, unsigned long long* stat, cudaStream_t s);
cudaError_t ts_launch_flip(const int16_t* l2r, int16_t* r2l, int w, int h, uint32_t* key, cudaStream_t s);
cudaError_t ts_launch_filter_speckles(int16_t* img, int w, int h, int newVal, int maxSize, int maxDiff, int* labels, int* sizes, cudaStream_t s);
int ts_filter_speckles_launches(int w, int h);
cudaError_t ts_launch_extract_mask(const int16_t* disp, uint8_t* mask, int w, int h, int thValid, cudaStream_t s);
cudaError_t ts_launch_upscale_mask(const uint8_t* m, int w, int h, uint8_t* m2, int w2, int h2, cudaStream_t s);
cudaError_t ts_launch_resize_area_u8(const uint8_t* src, int sw, int sh, int ch, int f, uint8_t* dst, int dw, int dh, cudaStream_t s);
cudaError_t ts_launch_fill_i16(int16_t* p, size_t n, int16_t v, cudaStream_t s);

namespace {

struct DevBuf {
	void* p = nullptr; size_t cap = 0;
	cudaError_t reserve(size_t n) {
		if (n <= cap) return cudaSuccess;
		if (p) cudaFree(p);
		p = nullptr; cap = 0;
		cudaError_t e = cudaMalloc(&p, n);
		if (e == cudaSuccess) cap = n;
		return e;
	}
	void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
	template <typename T> T* as() const { return (T*)p; }
};

void mul33(const double* A, const double* B, double* C) {
	double T[9];
	for (int i=0;i<3;++i) for (int j=0;j<3;++j) T[i*3+j] = A[i*3]*B[j] + A[i*3+1]*B[3+j] + A[i*3+2]*B[6+j];
	memcpy(C, T, sizeof(T));
}
void mul31(const double* A, const double* v, double* r) {
	double t[3];
	for (int i=0;i<3;++i) t[i] = A[i*3]*v[0] + A[i*3+1]*v[1] + A[i*3+2]*v[2];
	memcpy(r, t, sizeof(t));
}
void transpose33(const double* A, double* T) {
	double R[9];
	for (int i=0;i<3;++i) for (int j=0;j<3;++j) R[j*3+i] = A[i*3+j];
	memcpy(T, R, sizeof(R));
}
void inv33(const double* A, double* I) {
	const double a=A[0],b=A[1],c=A[2],d=A[3],e=A[4],f=A[5],g=A[6],h=A[7],i=A[8];
	const double id = 1.0/(a*(e*i-f*h) - b*(d*i-f*g) + c*(d*h-e*g));
	double R[9] = {(e*i-f*h)*id, (c*h-b*i)*id, (b*f-c*e)*id, (f*g-d*i)*id, (a*i-c*g)*id, (c*d-a*f)*id, (d*h-e*g)*id, (b*g-a*h)*id, (a*e-b*d)*id};
	memcpy(I, R, sizeof(R));
}
// Camera::ScaleK (libs/MVS/Camera.h:160-173)
void scaleK(const double* K, int sw, int sh, int dw, int dh, double* Ko) {
	const double sx = (double)dw/sw, sy = (double)dh/sh;
	Ko[0] = K[0]*sx; Ko[1] = K[1]*sx; Ko[2] = (K[2]+0.5)*sx-0.5;
	Ko[3] = 0; Ko[4] = K[4]*sy; Ko[5] = (K[5]+0.5)*sy-0.5;
	Ko[6] = 0; Ko[7] = 0; Ko[8] = 1;
}
inline float d2r(float d) { return d*(3.14159265358979323846f/180.f); }

// a view whose image (and optional depth-map) pointers are device pointers, pitch in floats
struct DView {
	const float* img; int w, h, pitch;
	double K[9], R[9], C[3];
	const float* dmap; int dw, dh, dpitch;
	double Kd[9], Rd[9], Cd[3];
};

} // namespace

struct b200mvs_ctx {
	int device = 0;
	b200mvs_params prm;
	std::string err;
	cudaStream_t stream = nullptr;
	cudaEvent_t ev0 = nullptr, ev1 = nullptr;
	// grow-only device scratch
	std::vector<DevBuf> imgs, dmaps, img8;    // staged images / depth-maps / 8-bit colour images (host API; gray images converted on the device)
	std::vector<DevBuf> pyr;                  // per-view pyramid levels (all levels packed)
	DevBuf plane, cost, best, prior, lowPlane;
	DevBuf dDepth, dNormal, dConf, dViews;    // level scratch / staging of the maps (host API)
	DevBuf mapD, mapN;                        // full-resolution in/out maps (host API)
	DevBuf sgL, sgC, sgR, sgPx, sgCosts, sgAccums, sgAccums2, sgDisp, sgCost, sgMax; // SGM staging / scratch
	// wave-front aggregation: cached schedule of the last (size, mode) and its scratch
	struct FrontPass { FrontLaunch launch; DevBuf items, need; int nItems = 0; };   // launch.items is emptied once uploaded
	std::vector<FrontPass> sgFront; int sgFrontKey[6] = {0, 0, 0, 0, 0, 0};
	DevBuf sgFrontCtl, sgFrontState, sgFrontMeta;
	cudaStream_t sgSide[7] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // side streams of the ragged aggregation
	cudaEvent_t sgJoin[7] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr}, sgFork = nullptr;
	const void* sgLastPx = nullptr; uint64_t sgLastNum = 0; // pixel map / size of the volume in sgAccums (b200mvs_sgm_refine_device check)
	bool sgFrontRan = false;                  // the last match aggregated with the wave-front kernel
	// coarse-to-fine SGM (b200mvs_sgm_match_tsgm_device): pyramid level images, range-map scratch, pixel map, level maps
	DevBuf tsLG, tsRG, tsLC, tsRC, tsRange, tsScratch, tsStat, tsPx, tsDisp, tsMask, tsLab, tsCost;
	DevBuf fltZ, fltIn, fltOutD, fltOutC;     // FilterDepthMap: z-buffer keys, staged maps (host API), outputs
	DevBuf ppA, ppB, ppD, ppN, ppC;           // RemoveSmallSegments labels/sizes, GapInterpolation temporaries, staging
	DevBuf ppK, ppArcs, ppPatch;              // RemoveSmallSegments: seed keys, one-way edges (+ counter), patched segment sizes
	b200mvs_debug dbg;                        // diagnostic switches (b200mvs_set_debug); all zero = the shipped kernels
	const uint8_t* mask = nullptr; int maskW = 0, maskH = 0, maskPitch = 0; // ignore-mask of the reference view (device) or null
	DevBuf maskBuf, maskLevel;                // staged host mask, mask of the current pyramid level
	DevBuf refPad;                            // 16-byte aligned copy of a reference image whose pitch TMA cannot address
	CUtensorMap tmapRef;                      // descriptor of the current level's reference image
	bool tmapValid = false;
	std::vector<cudaEvent_t> sweepEv;         // event pairs around the sweep launches (stats only)
	int nSweepEv = 0; bool timeSweeps = false;
	int launches = 0;
	// state of an enqueued b200mvs_estimate_async call
	bool pending = false; uint64_t pendH2D = 0, pendD2H = 0; int pendLevels = 1;
	std::chrono::steady_clock::time_point t0;
};

namespace {

int fail(b200mvs_ctx* c, int code, const char* what, cudaError_t e = cudaSuccess) {
	if (c) {
		c->err = what;
		if (e != cudaSuccess) { c->err += ": "; c->err += cudaGetErrorString(e); }
	}
	return code;
}
#define CK(call) do { cudaError_t _e = (call); if (_e != cudaSuccess) return fail(ctx, B200MVS_ERR_CUDA, #call, _e); } while (0)

// fill the kernel parameter block for one resolution level (DepthEstimator ctor constants,
// libs/MVS/DepthMap.cpp:361-412, and ViewData::Init, libs/MVS/DepthMap.h:175-185)
void build_params(const b200mvs_params& o, const DView* v, int nViews, float dMin, float dMax,
	const float* lowres, float4* plane, float* cost, uint32_t* best, PMParams& P, bool& geom)
{
	memset(&P, 0, sizeof(P));
	P.img0 = v[0].img; P.W = v[0].w; P.H = v[0].h; P.pitch0 = v[0].pitch;
	P.nViews = nViews-1;
	const double* K = v[0].K;
	P.ifx = (float)(1.0/K[0]); P.sk = (float)(-K[1]/(K[0]*K[4])); P.ox = (float)((K[1]*K[5]-K[2]*K[4])/(K[0]*K[4]));
	P.ify = (float)(1.0/K[4]); P.oy = (float)(-K[5]/K[4]);
	P.ox0 = (float)(-K[2]/K[0]);
	P.dMin = dMin; P.dMax = dMax; P.dMinSqr = std::sqrt(dMin); P.dMaxSqr = std::sqrt(dMax);
	P.keep = o.fNCCThresholdKeep;
	P.thMagnitudeSq = o.fDescriptorMinMagnitudeThreshold > 0 ? o.fDescriptorMinMagnitudeThreshold*o.fDescriptorMinMagnitudeThreshold : -1.f;
	P.thConfSmall = o.fNCCThresholdKeep*0.66f; P.thConfBig = o.fNCCThresholdKeep*0.9f;
	P.thConfRand = o.fNCCThresholdKeep*1.1f; P.thRobust = o.fNCCThresholdKeep*4.f/3.f;
	P.smoothBonusDepth = 1.f-o.fRandomSmoothBonus; P.smoothBonusNormal = (1.f-o.fRandomSmoothBonus)*0.96f;
	P.smoothSigmaDepth = -1.f/(2.f*o.fRandomSmoothDepth*o.fRandomSmoothDepth);
	P.smoothSigmaNormal = -1.f/(2.f*d2r(o.fRandomSmoothNormal)*d2r(o.fRandomSmoothNormal));
	P.depthRatio = o.fRandomDepthRatio; P.angle1Range = d2r(o.fRandomAngle1Range); P.angle2Range = d2r(o.fRandomAngle2Range);
	P.geomWeight = o.fEstimationGeometricWeight;
	P.nRandomIters = o.nRandomIters; P.propagation = o.nPropagation;
	P.farRings = o.nPropagationFar; P.evalCap = o.nEvalCap; P.skipUnchanged = 0; // the estimate call turns the changed-flag rule on; building blocks keep costs unsigned
	P.seed = o.seed;
	P.lowres = lowres; P.plane = plane; P.cost = cost; P.bestViews = best;
	double RrT[9], Hr[9], KrRr[9];
	transpose33(v[0].R, RrT);
	inv33(v[0].K, Hr);
	mul33(v[0].K, v[0].R, KrRr);
	geom = false;
	for (int i = 1; i < nViews; ++i) {
		PMView& V = P.views[i-1];
		double KR[9], Hl[9], A[9], dC[3], Hm[3];
		mul33(v[i].K, v[i].R, KR);
		mul33(KR, RrT, Hl);
		mul33(Hl, Hr, A);
		for (int k=0;k<3;++k) dC[k] = v[0].C[k]-v[i].C[k];
		mul31(KR, dC, Hm);
		for (int k=0;k<9;++k) V.A[k] = (float)A[k];
		for (int k=0;k<3;++k) V.Hm[k] = (float)Hm[k];
		V.img = v[i].img; V.w = v[i].w; V.h = v[i].h; V.pitch = v[i].pitch;
		V.dmap = v[i].dmap; V.dw = v[i].dw; V.dh = v[i].dh; V.dpitch = v[i].dpitch;
		if (v[i].dmap) {
			geom = true;
			double KdRd[9], T[9], t[3], RdT[9], iKd[9];
			mul33(v[i].Kd, v[i].Rd, KdRd);
			mul33(KdRd, RrT, T);
			for (int k=0;k<9;++k) V.Tl[k] = (float)T[k];
			for (int k=0;k<3;++k) dC[k] = v[0].C[k]-v[i].Cd[k];
			mul31(KdRd, dC, t);
			for (int k=0;k<3;++k) V.Tm[k] = (float)t[k];
			transpose33(v[i].Rd, RdT);
			inv33(v[i].Kd, iKd);
			mul33(KrRr, RdT, T); mul33(T, iKd, T);
			for (int k=0;k<9;++k) V.Tr[k] = (float)T[k];
			for (int k=0;k<3;++k) dC[k] = v[i].Cd[k]-v[0].C[k];
			mul31(KrRr, dC, t);
			for (int k=0;k<3;++k) V.Tn[k] = (float)t[k];
		}
	}
}

int check_views(b200mvs_ctx* ctx, const b200mvs_view* views, int nViews) {
	if (!ctx) return B200MVS_ERR_ARG;
	if (!views || nViews < 2 || nViews > B200MVS_MAX_VIEWS+1)
		return fail(ctx, B200MVS_ERR_ARG, "need 2..33 views (reference first)");
	for (int i = 0; i < nViews; ++i) {
		if ((!views[i].image && !views[i].image8) || views[i].width < 2*PM_HALF+2 || views[i].height < 2*PM_HALF+2)
			return fail(ctx, B200MVS_ERR_ARG, "view without image or image too small");
		if (!views[i].image && views[i].channels8 != 3 && views[i].channels8 != 4)
			return fail(ctx, B200MVS_ERR_ARG, "8-bit image needs 3 or 4 channels");
	}
	return B200MVS_OK;
}

void to_dview(const b200mvs_view& s, const float* img, int pitch, const float* dmap, int dpitch, DView& d) {
	d.img = img; d.w = s.width; d.h = s.height; d.pitch = pitch;
	memcpy(d.K, s.K, sizeof(d.K)); memcpy(d.R, s.R, sizeof(d.R)); memcpy(d.C, s.C, sizeof(d.C));
	d.dmap = dmap; d.dw = s.dwidth; d.dh = s.dheight; d.dpitch = dpitch;
	memcpy(d.Kd, s.Kd, sizeof(d.Kd)); memcpy(d.Rd, s.Rd, sizeof(d.Rd)); memcpy(d.Cd, s.Cd, sizeof(d.Cd));
}

inline int cvRoundI(double v) { return (int)std::nearbyint(v); }

// The engine's red-black schedule for nEstimationIters reference iterations (DESIGN.md §2): nSweeps red-black sweeps with nR
// refinement tries each.  nSweepsPerIter > 0 pins it (nSweeps = nSweepsPerIter x iterations, nR = ceil(nRandomIters /
// nSweepsPerIter)); 0 (default) = max(8, ceil(1.5 x iterations)) sweeps sharing the reference's nRandomIters x iterations
// tries.  A geometric pass (one reference iteration on a converged estimate) is 2 sweeps (or nSweepsPerIter).
void engine_schedule(const b200mvs_params& o, bool geometric, int& nSweeps, int& nR) {
	const int I = std::max(0, o.nEstimationIters);
	if (o.nSweepsPerIter > 0 || geometric) {
		const int spi = o.nSweepsPerIter > 0 ? o.nSweepsPerIter : 2;
		nSweeps = geometric ? spi : spi*I;
		nR = (o.nRandomIters+spi-1)/spi;
	} else {
		nSweeps = I > 0 ? std::max(8, (3*I+1)/2) : 0;
		nR = nSweeps > 0 ? (o.nRandomIters*I+nSweeps-1)/nSweeps : 0;
	}
}

// cuTensorMapEncodeTiled through the runtime (no link against libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
	const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn() {
	static EncodeTiledFn fn = nullptr; static bool tried = false;
	if (!tried) {
		tried = true;
		void* p = nullptr; cudaDriverEntryPointQueryResult q;
		if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
			fn = (EncodeTiledFn)p;
	}
	return fn;
}

// TMA descriptor of the reference image of one level: 2-D float tensor {W, H}, box = the tile a CTA
// of the sweep kernel stages (72 x 16).  TMA needs a 16-byte aligned base and row pitch; an image that
// does not satisfy this (odd width, cv::Mat ROI) is first copied to an aligned scratch image.
int prepare_ref_tmap(b200mvs_ctx* ctx, const DView& ref, cudaStream_t s) {
	ctx->tmapValid = false;
	EncodeTiledFn enc = ctx->dbg.noTMA ? nullptr : encode_tiled_fn();
	if (!enc) return B200MVS_OK;
	const float* base = ref.img; size_t pitchB = (size_t)ref.pitch*4;
	if (((uintptr_t)base & 15) || (pitchB & 15)) {
		pitchB = (((size_t)ref.w*4)+15)&~(size_t)15;
		CK(ctx->refPad.reserve(pitchB*ref.h));
		CK(cudaMemcpy2DAsync(ctx->refPad.p, pitchB, ref.img, (size_t)ref.pitch*4, (size_t)ref.w*4, ref.h, cudaMemcpyDeviceToDevice, s));
		base = ctx->refPad.as<float>();
	}
	int bw, bh; pm_tma_box(&bw, &bh);
	const cuuint64_t dims[2] = {(cuuint64_t)ref.w, (cuuint64_t)ref.h};
	const cuuint64_t strides[1] = {(cuuint64_t)pitchB};
	const cuuint32_t box[2] = {(cuuint32_t)bw, (cuuint32_t)bh};
	const cuuint32_t estr[2] = {1, 1};
	const CUresult r = enc(&ctx->tmapRef, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, dims, strides, box, estr,
		CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
	ctx->tmapValid = (r == CUDA_SUCCESS);
	return B200MVS_OK;
}

int launch_sweep_timed(b200mvs_ctx* ctx, const PMParams& P, bool geom, cudaStream_t s) {
	if (ctx->timeSweeps) {
		while ((int)ctx->sweepEv.size() < 2*(ctx->nSweepEv+1)) {
			cudaEvent_t e; CK(cudaEventCreate(&e)); ctx->sweepEv.push_back(e);
		}
		CK(cudaEventRecord(ctx->sweepEv[2*ctx->nSweepEv], s));
	}
	CK(pm_launch_sweep(P, ctx->tmapValid ? &ctx->tmapRef : nullptr, !ctx->dbg.scalarTaps, geom, ctx->dbg.sweepFourCtas != 0, s)); ++ctx->launches;
	if (ctx->timeSweeps) {
		CK(cudaEventRecord(ctx->sweepEv[2*ctx->nSweepEv+1], s));
		++ctx->nSweepEv;
	}
	return B200MVS_OK;
}

// The whole EstimateDepthMap on device-resident views.  d_depth/d_normal hold the initial
// estimate (full resolution) and receive the result together with d_conf / d_views.
int estimate_on_device(b200mvs_ctx* ctx, const DView* views, int nViews, float dMin, float dMax, int nGeometricIter,
	float* d_depth, float* d_normal, float* d_conf, uint32_t* d_views, cudaStream_t s)
{
	const b200mvs_params& o = ctx->prm;
	const int W = views[0].w, H = views[0].h;
	const bool geometric = nGeometricIter >= 0;
	int nSweepsPhoto, nRPhoto, nSweeps, nR;
	engine_schedule(o, false, nSweepsPhoto, nRPhoto);
	engine_schedule(o, geometric, nSweeps, nR);
	// Philox phase of the first sweep of this call: photometric sweeps 0 .. nSweepsPhoto-1, then the geometric passes
	const int sweepBase = geometric ? nSweepsPhoto + nGeometricIter*nSweeps : 0;
	const int totalScale = !geometric ? std::max(0, o.nSubResolutionLevels) : 0;
	const size_t P0 = (size_t)W*H;
	if (ctx->mask && (ctx->maskW != W || ctx->maskH != H))
		return fail(ctx, B200MVS_ERR_ARG, "ignore-mask size differs from the reference image");
	CK(ctx->plane.reserve(P0*sizeof(float4)));
	CK(ctx->cost.reserve(P0*sizeof(float)));
	CK(ctx->best.reserve(P0*sizeof(uint32_t)));
	if (totalScale > 0) {
		CK(ctx->prior.reserve(P0*sizeof(float)));
		CK(ctx->lowPlane.reserve((size_t)(W/2+2)*(H/2+2)*sizeof(float4)));
		if (ctx->mask) CK(ctx->maskLevel.reserve((size_t)(W/2+2)*(H/2+2)));
		if ((int)ctx->pyr.size() < nViews) ctx->pyr.resize(nViews);
		// level 1 is the largest pyramid level: size the buffers once, so that no level re-allocates mid-stream
		for (int i = 0; i < nViews; ++i) {
			const size_t dw = (size_t)cvRoundI(views[i].w*0.5), dh = (size_t)cvRoundI(views[i].h*0.5);
			CK(ctx->pyr[i].reserve(dw*dh*sizeof(float)*(views[i].dmap ? 2 : 1)));
		}
	}
	float4* plane = ctx->plane.as<float4>();
	float* cost = ctx->cost.as<float>();
	uint32_t* best = ctx->best.as<uint32_t>();
	int lowW = 0, lowH = 0;
	for (int sc = totalScale; sc >= 0; --sc) {
		// ScaleDepthData (SceneDensify.cpp:578-601): INTER_AREA images, rescaled K
		std::vector<DView> lv(views, views+nViews);
		if (sc > 0) {
			const double scale = 1.0/(double)(1<<sc);
			for (int i = 0; i < nViews; ++i) {
				const int dw = cvRoundI(views[i].w*scale), dh = cvRoundI(views[i].h*scale);
				if (dw < 2*PM_HALF+2 || dh < 2*PM_HALF+2)
					return fail(ctx, B200MVS_ERR_ARG, "image too small for nSubResolutionLevels");
				const size_t need = (size_t)dw*dh*sizeof(float)*(views[i].dmap ? 2 : 1);
				CK(ctx->pyr[i].reserve(need));
				float* im = ctx->pyr[i].as<float>();
				CK(rs_launch_area(views[i].img, views[i].w, views[i].h, views[i].pitch, im, dw, dh, 1.0/scale, 1.0/scale, s)); ++ctx->launches;
				lv[i].img = im; lv[i].w = dw; lv[i].h = dh; lv[i].pitch = dw;
				scaleK(views[i].K, views[i].w, views[i].h, dw, dh, lv[i].K);
				if (views[i].dmap) {
					float* dm = im + (size_t)dw*dh;
					CK(rs_launch_area(views[i].dmap, views[i].dw, views[i].dh, views[i].dpitch, dm, dw, dh, 0, 0, s)); ++ctx->launches;
					lv[i].dmap = dm; lv[i].dw = dw; lv[i].dh = dh; lv[i].dpitch = dw;
					scaleK(views[i].Kd, views[i].dw, views[i].dh, dw, dh, lv[i].Kd);
				}
			}
		}
		const int w = lv[0].w, h = lv[0].h;
		{ const int rc = prepare_ref_tmap(ctx, lv[0], s); if (rc) return rc; }
		const float* lowres = nullptr;
		if (sc != totalScale) {
			// depth LINEAR / normal NEAREST up-sampling of the coarser level; the up-sampled
			// depth is also the prior of this level (SceneDensify.cpp:660-664)
			CK(rs_launch_plane_up(ctx->lowPlane.as<float4>(), lowW, lowH, plane, ctx->prior.as<float>(), w, h, ctx->mask != nullptr, s)); ++ctx->launches;
			lowres = ctx->prior.as<float>();
		} else if (sc == 0) {
			CK(pm_launch_pack((int)P0, d_depth, d_normal, plane, s)); ++ctx->launches;
		} else {
			// coarsest level: the caller's initial estimate, NEAREST down-sampled
			CK(ctx->dDepth.reserve((size_t)w*h*sizeof(float)));
			CK(ctx->dNormal.reserve((size_t)w*h*3*sizeof(float)));
			CK(rs_launch_nearest(d_depth, W, H, 1, ctx->dDepth.as<float>(), w, h, (double)(1<<sc), (double)(1<<sc), s));
			CK(rs_launch_nearest(d_normal, W, H, 3, ctx->dNormal.as<float>(), w, h, (double)(1<<sc), (double)(1<<sc), s));
			CK(pm_launch_pack(w*h, ctx->dDepth.as<float>(), ctx->dNormal.as<float>(), plane, s)); ctx->launches += 3;
		}
		PMParams P; bool geom;
		build_params(o, lv.data(), nViews, dMin, dMax, lowres, plane, cost, best, P, geom);
		P.nRandomIters = nR;
		P.skipUnchanged = o.bSkipUnchanged ? 1 : 0;
		P.tma = ctx->tmapValid ? 1 : 0;
		if (ctx->mask) {
			// the mask of this level: cv::resize(..., INTER_NEAREST) of the full-resolution mask (DepthMap.cpp:309)
			if (sc > 0) {
				CK(rs_launch_nearest_u8(ctx->mask, W, H, ctx->maskPitch, ctx->maskLevel.as<uint8_t>(), w, h, s)); ++ctx->launches;
				P.mask = ctx->maskLevel.as<uint8_t>(); P.maskPitch = w;
			} else { P.mask = ctx->mask; P.maskPitch = ctx->maskPitch; }
		}
		CK(pm_launch_score(P, !ctx->dbg.scalarTaps, geom, s)); ++ctx->launches;
		for (int k = 0; k < nSweeps; ++k) {
			P.sweep = sweepBase+k;
			for (int colour = 0; colour < 2; ++colour) {
				P.colour = colour;
				{ const int rc = launch_sweep_timed(ctx, P, geom, s); if (rc) return rc; }
			}
		}
		if (sc > 0) {
			CK(cudaMemcpyAsync(ctx->lowPlane.p, plane, (size_t)w*h*sizeof(float4), cudaMemcpyDeviceToDevice, s));
			lowW = w; lowH = h;
		}
	}
	float keep = o.fNCCThresholdKeep;
	if (nGeometricIter < 0 && o.nEstimationGeometricIters)
		keep *= 1.333f;
	CK(pm_launch_finalize((int)P0, keep, plane, cost, best, d_depth, d_normal, d_conf, d_views, s)); ++ctx->launches;
	return B200MVS_OK;
}

// SGM path aggregation with the wave-front kernel (sgm_front.cu).  Pass layouts (b200mvs_debug.frontLayout, 0 = auto = 1):
//   1 two tilted fronts f = +-(x + 2y): {right, right-down, down, left-down} and {left, left-up, up, right-up};
//   2 four straight fronts: top-down {down, right-down, left-down}, bottom-up {up, right-up, left-up}, left-right, right-left;
//   3 eight passes of one direction each (the traffic of the per-direction kernels with the new step).
// Unless frontSerial is set, consecutive passes share a launch: pass 2j accumulates into the caller's volume, pass 2j+1 into a
// second one (ctx->sgAccums2), and `twoVolumes` tells the caller to add them (the winner-takes-all kernel does).
int sgm_aggregate_fronts(b200mvs_ctx* ctx, const SGMParams& P, int num, cudaStream_t s, bool& twoVolumes) {
	const b200mvs_debug& D = ctx->dbg;
	const int layout = std::min(std::max(D.frontLayout-1, 0), 2);
	const bool concurrent = !D.frontSerial;
	const int FB = D.frontBlock > 0 ? D.frontBlock : 32;   // measured: profiles/sgm_variants_r02f.txt (64: 4 % faster, a third more DRAM traffic at lag 2)
	// frontLag = lag + 1.  The sub-cell dependencies make every lag legal; measured for 1914x1074x128 (profiles/sgm_variants_r02f.txt,
	// profiles/front_traffic_*_r02.csv): lag 2: 2.6 ms with 6.4 GB of DRAM traffic (the window of blocks between a block's first and
	// last phase exceeds the L2); lag 1: 2.9 ms with 2.0 GB — the algorithmic volume; lag 0: 2.2 GB but 5.1 ms (the resident warps all
	// hold items of one block and wait for each other).  Default: lag 1.
	const int lag = D.frontLag > 0 ? D.frontLag-1 : 1;
	const int vw = P.vw, vh = P.vh;
	// sub-cell width: one lane polls one counter, and a band at an image corner can span the whole width: at most 30 sub-cell columns
	const int SW = std::max(D.frontSubCell >= 16 ? D.frontSubCell : FRONT_SW, (vw+29)/30);
	const int key[6] = {vw, vh, layout, FB, lag | (SW<<8), concurrent ? 2 : 1};
	if (memcmp(key, ctx->sgFrontKey, sizeof(key)) != 0) {
		for (auto& fp: ctx->sgFront) { fp.items.release(); fp.need.release(); }
		ctx->sgFront.clear();
		std::vector<FrontLaunch> plan = sgm_front_plan(vw, vh, layout, concurrent, FB, lag, SW);
		ctx->sgFront.resize(plan.size());
		for (size_t i = 0; i < plan.size(); ++i) {
			b200mvs_ctx::FrontPass& fp = ctx->sgFront[i];
			CK(fp.items.reserve(plan[i].items.size()*sizeof(FrontItem)));
			CK(cudaMemcpyAsync(fp.items.p, plan[i].items.data(), plan[i].items.size()*sizeof(FrontItem), cudaMemcpyHostToDevice, s));
			CK(fp.need.reserve(std::max<size_t>(1, plan[i].cellNeed.size())*sizeof(int)));
			CK(cudaMemcpyAsync(fp.need.p, plan[i].cellNeed.data(), plan[i].cellNeed.size()*sizeof(int), cudaMemcpyHostToDevice, s));
			CK(cudaStreamSynchronize(s)); // the pageable source vectors are released below
			fp.nItems = (int)plan[i].items.size();
			plan[i].items.clear(); plan[i].items.shrink_to_fit(); plan[i].cellNeed.clear(); plan[i].cellNeed.shrink_to_fit();
			fp.launch = plan[i];
		}
		CK(cudaStreamSynchronize(s)); // the pageable source vectors die with `plan`
		memcpy(ctx->sgFrontKey, key, sizeof(key));
	}
	twoVolumes = false;
	for (auto& fp: ctx->sgFront) twoVolumes |= fp.launch.nPasses > 1;
	uint16_t* second = nullptr;
	if (twoVolumes) {
		CK(ctx->sgAccums2.reserve((size_t)vw*vh*num*sizeof(uint16_t)));
		second = ctx->sgAccums2.as<uint16_t>();
	}
	const int maxPaths = vw+vh+8;
	int maxCtl = 0;
	for (auto& fp: ctx->sgFront) maxCtl = std::max(maxCtl, fp.launch.nChains + fp.launch.nCells);
	CK(ctx->sgFrontCtl.reserve((size_t)(4+maxCtl)*sizeof(int)));
	CK(ctx->sgFrontState.reserve((size_t)8*maxPaths*num*sizeof(uint16_t)));
	CK(ctx->sgFrontMeta.reserve((size_t)8*maxPaths*sizeof(float2)));
	int* ctl = ctx->sgFrontCtl.as<int>();
	// resident CTAs: the queue needs no particular number; frontCtas = CTAs per SM, frontDepth = ring slots per warp (8 default, 4)
	const int pd = D.frontDepth == 4 ? 4 : 8;
	int sms = 148; cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
	const int perSm = std::min(sgm_front_blocks_per_sm(num, pd), D.frontCtas > 0 ? D.frontCtas : 2);
	const int blocks = sms*perSm;
	const int FBeff = layout == 2 ? (1<<28) : FB;
	for (size_t i = 0; i < ctx->sgFront.size(); ++i) {
		b200mvs_ctx::FrontPass& fp = ctx->sgFront[i];
		const FrontLaunch& L = fp.launch;
		// [ticket, error, -, - | progress | cellDone]; the error word survives the launches of one call
		if (i == 0) CK(cudaMemsetAsync(ctl, 0, (size_t)(4+maxCtl)*sizeof(int), s));
		else { CK(cudaMemsetAsync(ctl, 0, sizeof(int), s)); CK(cudaMemsetAsync(ctl+4, 0, (size_t)maxCtl*sizeof(int), s)); }
		FrontArgs A; memset(&A, 0, sizeof(A));
		A.items = fp.items.as<FrontItem>(); A.nItems = fp.nItems;
		A.ticket = ctl; A.error = ctl+1; A.progress = ctl+4; A.cellDone = ctl+4+L.nChains; A.cellNeed = fp.need.as<int>();
		A.state = ctx->sgFrontState.as<uint16_t>(); A.meta = ctx->sgFrontMeta.as<float2>(); A.maxPaths = maxPaths;
		A.FB = FBeff; A.num = num;
		for (int p = 0; p < L.nPasses; ++p) {
			A.fa[p] = L.pass[p].fa; A.fb[p] = L.pass[p].fb; A.fc[p] = L.fc[p];
			A.storePhase0[p] = i == 0 ? 1 : 0;
			A.sum[p] = p == 0 ? P.accums : second;
		}
		CK(sgm_front_launch(P, A, blocks, pd, s)); ++ctx->launches;
	}
	return B200MVS_OK;
}

} // namespace

extern "C" {

int b200mvs_device_count(void) {
	int n = 0;
	if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
	return n;
}

void b200mvs_default_params(b200mvs_params* p) {
	p->nEstimationIters = 3; p->nEstimationGeometricIters = 2; p->nRandomIters = 6; p->nSubResolutionLevels = 2;
	p->fNCCThresholdKeep = 0.9f; p->fDescriptorMinMagnitudeThreshold = 0.02f;
	p->fRandomDepthRatio = 0.003f; p->fRandomAngle1Range = 16.f; p->fRandomAngle2Range = 10.f;
	p->fRandomSmoothDepth = 0.02f; p->fRandomSmoothNormal = 13.f; p->fRandomSmoothBonus = 0.93f;
	p->fEstimationGeometricWeight = 0.1f;
	p->nSweepsPerIter = 0; p->nPropagation = 4; p->seed = 1234u;
	p->nPropagationFar = 2; p->bSkipUnchanged = 1; p->nEvalCap = 0;
}

/* bumped whenever a struct of b200mvs.h changes layout; bindings compare it (and the struct sizes) at load time */
int b200mvs_abi_version(void) { return B200MVS_ABI_VERSION; }
size_t b200mvs_sizeof(int what) {
	switch (what) {
	case 0: return sizeof(b200mvs_view);
	case 1: return sizeof(b200mvs_params);
	case 2: return sizeof(b200mvs_stats);
	case 3: return sizeof(b200mvs_job);
	case 4: return sizeof(b200mvs_sgm_pixel);
	case 5: return sizeof(b200mvs_sgm_params);
	case 6: return sizeof(b200mvs_dmap);
	case 7: return sizeof(b200mvs_filter_params);
	case 8: return sizeof(b200mvs_debug);
	default: return 0;
	}
}

int b200mvs_create(int device, b200mvs_ctx** out) {
	if (!out) return B200MVS_ERR_ARG;
	*out = nullptr;
	int n = 0;
	if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0)
		return B200MVS_ERR_NOGPU; // never falls back to a CPU path
	if (device < 0) device = 0;
	if (device >= n) return B200MVS_ERR_ARG;
	if (cudaSetDevice(device) != cudaSuccess) return B200MVS_ERR_CUDA;
	b200mvs_ctx* c = new b200mvs_ctx();
	c->device = device;
	b200mvs_default_params(&c->prm);
	memset(&c->dbg, 0, sizeof(c->dbg));
	// dynamic shared memory opt-in of the kernels on this device (per-device attributes; idempotent, thread-safe)
	if (pm_configure_device() != cudaSuccess || sgm_configure_device() != cudaSuccess || sgm_cost_tc_configure() != cudaSuccess) { delete c; return B200MVS_ERR_CUDA; }
	if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess ||
		cudaEventCreate(&c->ev0) != cudaSuccess || cudaEventCreate(&c->ev1) != cudaSuccess) {
		delete c;
		return B200MVS_ERR_CUDA;
	}
	*out = c;
	return B200MVS_OK;
}

int b200mvs_destroy(b200mvs_ctx* c) {
	if (!c) return B200MVS_ERR_ARG;
	cudaSetDevice(c->device);
	if (c->stream) cudaStreamSynchronize(c->stream); // an enqueued asynchronous call may still use the buffers
	for (auto& b: c->imgs) b.release();
	for (auto& b: c->dmaps) b.release();
	for (auto& b: c->img8) b.release();
	for (auto& b: c->pyr) b.release();
	c->refPad.release(); c->maskBuf.release(); c->maskLevel.release();
	for (auto e: c->sweepEv) cudaEventDestroy(e);
	c->sgL.release(); c->sgC.release(); c->sgR.release(); c->sgPx.release(); c->sgCosts.release(); c->sgAccums.release(); c->sgAccums2.release();
	c->sgDisp.release(); c->sgCost.release(); c->sgMax.release();
	for (DevBuf* b: {&c->tsLG, &c->tsRG, &c->tsLC, &c->tsRC, &c->tsRange, &c->tsScratch, &c->tsStat, &c->tsPx, &c->tsDisp, &c->tsMask, &c->tsLab, &c->tsCost})
		b->release();
	for (auto& fp: c->sgFront) { fp.items.release(); fp.need.release(); }
	c->sgFrontCtl.release(); c->sgFrontState.release(); c->sgFrontMeta.release();
	for (int i = 0; i < 7; ++i) { if (c->sgSide[i]) cudaStreamDestroy(c->sgSide[i]); if (c->sgJoin[i]) cudaEventDestroy(c->sgJoin[i]); }
	if (c->sgFork) cudaEventDestroy(c->sgFork);
	c->fltZ.release(); c->fltIn.release(); c->fltOutD.release(); c->fltOutC.release();
	c->ppA.release(); c->ppB.release(); c->ppD.release(); c->ppN.release(); c->ppC.release();
	c->ppK.release(); c->ppArcs.release(); c->ppPatch.release();
	c->plane.release(); c->cost.release(); c->best.release(); c->prior.release(); c->lowPlane.release();
	c->dDepth.release(); c->dNormal.release(); c->dConf.release(); c->dViews.release(); c->mapD.release(); c->mapN.release();
	if (c->ev0) cudaEventDestroy(c->ev0);
	if (c->ev1) cudaEventDestroy(c->ev1);
	if (c->stream) cudaStreamDestroy(c->stream);
	delete c;
	return B200MVS_OK;
}

int b200mvs_set_params(b200mvs_ctx* ctx, const b200mvs_params* p) {
	if (!ctx || !p) return B200MVS_ERR_ARG;
	if (p->nEstimationIters < 0 || p->nRandomIters < 0 || p->nSweepsPerIter < 0 || (p->nPropagation != 2 && p->nPropagation != 4) ||
		p->nPropagationFar < 0 || p->nPropagationFar > 3 || p->nEvalCap < 0 || p->nEvalCap > 15 || p->nSubResolutionLevels < 0 || !(p->fNCCThresholdKeep > 0))
		return fail(ctx, B200MVS_ERR_ARG, "invalid parameter block");
	ctx->prm = *p;
	return B200MVS_OK;
}

int b200mvs_set_debug(b200mvs_ctx* ctx, const b200mvs_debug* d) {
	if (!ctx) return B200MVS_ERR_ARG;
	if (d) ctx->dbg = *d; else memset(&ctx->dbg, 0, sizeof(ctx->dbg));
	return B200MVS_OK;
}

int b200mvs_get_schedule(const b200mvs_params* p, int geometric, int* nSweeps, int* nRefinePerSweep) {
	if (!p || !nSweeps || !nRefinePerSweep) return B200MVS_ERR_ARG;
	engine_schedule(*p, geometric != 0, *nSweeps, *nRefinePerSweep);
	return B200MVS_OK;
}

int b200mvs_set_ignore_mask(b200mvs_ctx* ctx, const uint8_t* mask, int width, int height, int stride_bytes, int on_device) {
	if (!ctx) return B200MVS_ERR_ARG;
	if (!mask) { ctx->mask = nullptr; ctx->maskW = ctx->maskH = ctx->maskPitch = 0; return B200MVS_OK; }
	if (width <= 0 || height <= 0 || (stride_bytes != 0 && stride_bytes < width))
		return fail(ctx, B200MVS_ERR_ARG, "ignore-mask: invalid size or stride");
	if (stride_bytes == 0) stride_bytes = width;
	CK(cudaSetDevice(ctx->device));
	if (on_device) { ctx->mask = mask; ctx->maskPitch = stride_bytes; }
	else {
		CK(ctx->maskBuf.reserve((size_t)width*height));
		CK(cudaMemcpy2DAsync(ctx->maskBuf.p, width, mask, stride_bytes, width, height, cudaMemcpyHostToDevice, ctx->stream));
		CK(cudaStreamSynchronize(ctx->stream)); // the caller's buffer may be released after the call
		ctx->mask = ctx->maskBuf.as<uint8_t>(); ctx->maskPitch = width;
	}
	ctx->maskW = width; ctx->maskH = height;
	return B200MVS_OK;
}

const char* b200mvs_last_error(const b200mvs_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int b200mvs_estimate_device(b200mvs_ctx* ctx, const b200mvs_view* views, int nViews, float dMin, float dMax, int nGeometricIter,
	float* depth, float* normal, float* conf, uint8_t* viewsMap, void* stream, b200mvs_stats* stats)
{
	int rc = check_views(ctx, views, nViews);
	if (rc) return rc;
	if (!depth || !normal || !conf || !(dMin > 0 && dMin < dMax))
		return fail(ctx, B200MVS_ERR_ARG, "null map pointer or invalid depth range");
	CK(cudaSetDevice(ctx->device));
	cudaStream_t s = stream ? (cudaStream_t)stream : ctx->stream;
	std::vector<DView> dv(nViews);
	ctx->launches = 0;
	for (int i = 0; i < nViews; ++i) {
		const float* img = views[i].image; int pitch = views[i].stride_bytes ? views[i].stride_bytes/4 : views[i].width;
		if (!img) {
			// 8-bit colour image resident in HBM: toGray into the context's scratch
			if ((int)ctx->imgs.size() < nViews) { ctx->imgs.resize(nViews); ctx->dmaps.resize(nViews); ctx->img8.resize(nViews); }
			CK(ctx->imgs[i].reserve((size_t)views[i].width*views[i].height*sizeof(float)));
			CK(rs_launch_to_gray(views[i].image8, views[i].width, views[i].height, views[i].stride8_bytes ? views[i].stride8_bytes : views[i].width*views[i].channels8,
				views[i].channels8, views[i].bgr8 != 0, ctx->imgs[i].as<float>(), views[i].width, s)); ++ctx->launches;
			img = ctx->imgs[i].as<float>(); pitch = views[i].width;
		}
		to_dview(views[i], img, pitch, views[i].depth, views[i].dstride_bytes ? views[i].dstride_bytes/4 : views[i].dwidth, dv[i]);
	}
	const auto t0 = std::chrono::steady_clock::now();
	ctx->nSweepEv = 0; ctx->timeSweeps = stats != nullptr;
	if (stats) CK(cudaEventRecord(ctx->ev0, s));
	rc = estimate_on_device(ctx, dv.data(), nViews, dMin, dMax, nGeometricIter, depth, normal, conf, (uint32_t*)viewsMap, s);
	if (rc) return rc;
	if (stats) {
		CK(cudaEventRecord(ctx->ev1, s));
		CK(cudaStreamSynchronize(s));
		float ms = 0; CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
		memset(stats, 0, sizeof(*stats));
		stats->ms_device = ms;
		stats->ms_total = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now()-t0).count();
		stats->kernel_launches = ctx->launches;
		stats->levels = (nGeometricIter < 0 ? ctx->prm.nSubResolutionLevels : 0)+1;
		for (int k = 0; k < ctx->nSweepEv; ++k) { float t = 0; CK(cudaEventElapsedTime(&t, ctx->sweepEv[2*k], ctx->sweepEv[2*k+1])); stats->ms_sweep_kernels += t; }
		stats->sweep_launches = ctx->nSweepEv;
		stats->tma_active = ctx->tmapValid ? 1 : 0;
	}
	return B200MVS_OK;
}

int b200mvs_estimate_async(b200mvs_ctx* ctx, const b200mvs_view* views, int nViews, float dMin, float dMax, int nGeometricIter,
	float* depth, float* normal, float* conf, uint8_t* viewsMap)
{
	int rc = check_views(ctx, views, nViews);
	if (rc) return rc;
	if (!depth || !normal || !conf || !(dMin > 0 && dMin < dMax))
		return fail(ctx, B200MVS_ERR_ARG, "null map pointer or invalid depth range");
	CK(cudaSetDevice(ctx->device));
	cudaStream_t s = ctx->stream;
	ctx->t0 = std::chrono::steady_clock::now();
	if ((int)ctx->imgs.size() < nViews) { ctx->imgs.resize(nViews); ctx->dmaps.resize(nViews); ctx->img8.resize(nViews); }
	std::vector<DView> dv(nViews);
	uint64_t h2d = 0, d2h = 0;
	ctx->launches = 0;
	for (int i = 0; i < nViews; ++i) {
		const b200mvs_view& v = views[i];
		const size_t row = (size_t)v.width*sizeof(float);
		CK(ctx->imgs[i].reserve(row*v.height));
		if (v.image) {
			CK(cudaMemcpy2DAsync(ctx->imgs[i].p, row, v.image, v.stride_bytes ? v.stride_bytes : row, row, v.height, cudaMemcpyHostToDevice, s));
			h2d += row*v.height;
		} else {
			// 8-bit colour image: upload channels8 bytes per pixel, convert on the device (toGray)
			const size_t row8 = (size_t)v.width*v.channels8;
			CK(ctx->img8[i].reserve(row8*v.height));
			CK(cudaMemcpy2DAsync(ctx->img8[i].p, row8, v.image8, v.stride8_bytes ? v.stride8_bytes : row8, row8, v.height, cudaMemcpyHostToDevice, s));
			h2d += row8*v.height;
			CK(rs_launch_to_gray(ctx->img8[i].as<uint8_t>(), v.width, v.height, (int)row8, v.channels8, v.bgr8 != 0, ctx->imgs[i].as<float>(), v.width, s)); ++ctx->launches;
		}
		const float* dm = nullptr;
		if (v.depth) {
			const size_t drow = (size_t)v.dwidth*sizeof(float);
			CK(ctx->dmaps[i].reserve(drow*v.dheight));
			CK(cudaMemcpy2DAsync(ctx->dmaps[i].p, drow, v.depth, v.dstride_bytes ? v.dstride_bytes : drow, drow, v.dheight, cudaMemcpyHostToDevice, s));
			h2d += drow*v.dheight;
			dm = ctx->dmaps[i].as<float>();
		}
		to_dview(v, ctx->imgs[i].as<float>(), v.width, dm, v.dwidth, dv[i]);
	}
	const size_t P0 = (size_t)views[0].width*views[0].height;
	DevBuf& dD = ctx->mapD; DevBuf& dN = ctx->mapN;
	CK(dD.reserve(P0*sizeof(float))); CK(dN.reserve(P0*3*sizeof(float)));
	CK(ctx->dConf.reserve(P0*sizeof(float))); CK(ctx->dViews.reserve(P0*sizeof(uint32_t)));
	CK(cudaMemcpyAsync(dD.p, depth, P0*sizeof(float), cudaMemcpyHostToDevice, s));
	CK(cudaMemcpyAsync(dN.p, normal, P0*3*sizeof(float), cudaMemcpyHostToDevice, s));
	h2d += P0*16;
	ctx->nSweepEv = 0; ctx->timeSweeps = true;
	CK(cudaEventRecord(ctx->ev0, s));
	rc = estimate_on_device(ctx, dv.data(), nViews, dMin, dMax, nGeometricIter, dD.as<float>(), dN.as<float>(),
		ctx->dConf.as<float>(), ctx->dViews.as<uint32_t>(), s);
	if (rc) return rc;
	CK(cudaEventRecord(ctx->ev1, s));
	CK(cudaMemcpyAsync(depth, dD.p, P0*sizeof(float), cudaMemcpyDeviceToHost, s));
	CK(cudaMemcpyAsync(normal, dN.p, P0*3*sizeof(float), cudaMemcpyDeviceToHost, s));
	CK(cudaMemcpyAsync(conf, ctx->dConf.p, P0*sizeof(float), cudaMemcpyDeviceToHost, s));
	d2h += P0*20;
	if (viewsMap) { CK(cudaMemcpyAsync(viewsMap, ctx->dViews.p, P0*4, cudaMemcpyDeviceToHost, s)); d2h += P0*4; }
	ctx->pendH2D = h2d; ctx->pendD2H = d2h; ctx->pendLevels = (nGeometricIter < 0 ? ctx->prm.nSubResolutionLevels : 0)+1;
	ctx->pending = true;
	return B200MVS_OK;
}

int b200mvs_sync(b200mvs_ctx* ctx, b200mvs_stats* stats) {
	if (!ctx) return B200MVS_ERR_ARG;
	CK(cudaSetDevice(ctx->device));
	CK(cudaStreamSynchronize(ctx->stream));
	if (stats) {
		memset(stats, 0, sizeof(*stats));
		if (ctx->pending) {
			float ms = 0; CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
			stats->ms_device = ms;
			stats->ms_total = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now()-ctx->t0).count();
			stats->bytes_h2d = ctx->pendH2D; stats->bytes_d2h = ctx->pendD2H;
			stats->kernel_launches = ctx->launches;
			stats->levels = ctx->pendLevels;
			for (int k = 0; k < ctx->nSweepEv; ++k) { float t = 0; CK(cudaEventElapsedTime(&t, ctx->sweepEv[2*k], ctx->sweepEv[2*k+1])); stats->ms_sweep_kernels += t; }
			stats->sweep_launches = ctx->nSweepEv;
			stats->tma_active = ctx->tmapValid ? 1 : 0;
		}
	}
	ctx->pending = false;
	return B200MVS_OK;
}

int b200mvs_estimate(b200mvs_ctx* ctx, const b200mvs_view* views, int nViews, float dMin, float dMax, int nGeometricIter,
	float* depth, float* normal, float* conf, uint8_t* viewsMap, b200mvs_stats* stats)
{
	const int rc = b200mvs_estimate_async(ctx, views, nViews, dMin, dMax, nGeometricIter, depth, normal, conf, viewsMap);
	if (rc) return rc;
	return b200mvs_sync(ctx, stats);
}

// Page-locks the caller's buffers for the duration of a batch: cudaMemcpyAsync from / to pageable memory blocks the host
// (and serialises the contexts); already pinned or unregistrable ranges are left alone.
namespace {
struct PinGuard {
	std::vector<void*> regs;
	void add(const void* p, size_t bytes) {
		if (!p || !bytes) return;
		if (cudaHostRegister((void*)p, bytes, cudaHostRegisterPortable) == cudaSuccess) regs.push_back((void*)p);
		else (void)cudaGetLastError(); // already registered (pinned by the caller, or shared between jobs): fine
	}
	~PinGuard() { for (void* p: regs) cudaHostUnregister(p); }
};
}

int b200mvs_estimate_batch(b200mvs_ctx** ctxs, int nCtx, b200mvs_job* jobs, int nJobs) {
	if (!ctxs || nCtx <= 0 || (!jobs && nJobs > 0) || nJobs < 0) return B200MVS_ERR_ARG;
	for (int k = 0; k < nCtx; ++k) if (!ctxs[k]) return B200MVS_ERR_ARG;
	PinGuard pin;
	for (int j = 0; j < nJobs; ++j) {
		const b200mvs_job& J = jobs[j];
		if (!J.views || J.nViews <= 0) continue;
		for (int i = 0; i < J.nViews; ++i) {
			const b200mvs_view& v = J.views[i];
			if (v.image) pin.add(v.image, (size_t)(v.stride_bytes ? v.stride_bytes : v.width*4)*v.height);
			else if (v.image8) pin.add(v.image8, (size_t)(v.stride8_bytes ? v.stride8_bytes : v.width*v.channels8)*v.height);
			if (v.depth) pin.add(v.depth, (size_t)(v.dstride_bytes ? v.dstride_bytes : v.dwidth*4)*v.dheight);
		}
		const size_t P0 = (size_t)J.views[0].width*J.views[0].height;
		pin.add(J.depth, P0*4); pin.add(J.normal, P0*12); pin.add(J.conf, P0*4); pin.add(J.viewsMap, P0*4);
	}
	int first = B200MVS_OK;
	std::vector<int> inflight(nCtx, -1); // job running on each context
	auto drain = [&](int k) {
		if (inflight[k] < 0) return;
		const int rc = b200mvs_sync(ctxs[k], nullptr);
		if (rc && !jobs[inflight[k]].status) jobs[inflight[k]].status = rc;
		if (jobs[inflight[k]].status && !first) first = jobs[inflight[k]].status;
		inflight[k] = -1;
	};
	for (int j = 0; j < nJobs; ++j) {
		const int k = j % nCtx;
		drain(k);
		b200mvs_job& J = jobs[j];
		J.status = b200mvs_estimate_async(ctxs[k], J.views, J.nViews, J.dMin, J.dMax, J.nGeometricIter, J.depth, J.normal, J.conf, J.viewsMap);
		if (J.status) { if (!first) first = J.status; continue; }
		inflight[k] = j;
	}
	for (int k = 0; k < nCtx; ++k) drain(k);
	return first;
}

// ---- building blocks ----------------------------------------------------------------------
int b200mvs_pm_pack(b200mvs_ctx* ctx, int width, int height, const float* depth, const float* normal, float* plane4, void* stream) {
	if (!ctx || !depth || !normal || !plane4) return B200MVS_ERR_ARG;
	CK(cudaSetDevice(ctx->device));
	CK(pm_launch_pack(width*height, depth, normal, (float4*)plane4, stream ? (cudaStream_t)stream : ctx->stream));
	return B200MVS_OK;
}
int b200mvs_pm_unpack(b200mvs_ctx* ctx, int width, int height, const float* plane4, float* depth, float* normal, void* stream) {
	if (!ctx || !depth || !normal || !plane4) return B200MVS_ERR_ARG;
	CK(cudaSetDevice(ctx->device));
	CK(pm_launch_unpack(width*height, (const float4*)plane4, depth, normal, stream ? (cudaStream_t)stream : ctx->stream));
	return B200MVS_OK;
}
static int block_params(b200mvs_ctx* ctx, const b200mvs_view* views, int nViews, float dMin, float dMax, const float* lowres,
	float* plane4, float* cost, cudaStream_t s, PMParams& P, bool& geom)
{
	int rc = check_views(ctx, views, nViews);
	if (rc) return rc;
	if (!plane4 || !cost) return fail(ctx, B200MVS_ERR_ARG, "null state pointer");
	for (int i = 0; i < nViews; ++i)
		if (!views[i].image) return fail(ctx, B200MVS_ERR_ARG, "the building blocks take float gray images");
	std::vector<DView> dv(nViews);
	for (int i = 0; i < nViews; ++i)
		to_dview(views[i], views[i].image, views[i].stride_bytes ? views[i].stride_bytes/4 : views[i].width,
			views[i].depth, views[i].dstride_bytes ? views[i].dstride_bytes/4 : views[i].dwidth, dv[i]);
	{ const int rc2 = prepare_ref_tmap(ctx, dv[0], s); if (rc2) return rc2; }
	build_params(ctx->prm, dv.data(), nViews, dMin, dMax, lowres, (float4*)plane4, cost, nullptr, P, geom);
	P.tma = ctx->tmapValid ? 1 : 0;
	return B200MVS_OK;
}
int b200mvs_pm_score(b200mvs_ctx* ctx, const b200mvs_view* views, int nViews, float dMin, float dMax,
	const float* lowres, float* plane4, float* cost, void* stream)
{
	PMParams P; bool geom;
	if (!ctx) return B200MVS_ERR_ARG;
	CK(cudaSetDevice(ctx->device));
	cudaStream_t s = stream ? (cudaStream_t)stream : ctx->stream;
	int rc = block_params(ctx, views, nViews, dMin, dMax, lowres, plane4, cost, s, P, geom);
	if (rc) return rc;
	CK(pm_launch_score(P, !ctx->dbg.scalarTaps, geom, s));
	return B200MVS_OK;
}
int b200mvs_pm_sweep(b200mvs_ctx* ctx, const b200mvs_view* views, int nViews, float dMin, float dMax,
	const float* lowres, int sweep, int half, int nRandomIters, float* plane4, float* cost, void* stream)
{
	PMParams P; bool geom;
	if (!ctx) return B200MVS_ERR_ARG;
	CK(cudaSetDevice(ctx->device));
	cudaStream_t s = stream ? (cudaStream_t)stream : ctx->stream;
	int rc = block_params(ctx, views, nViews, dMin, dMax, lowres, plane4, cost, s, P, geom);
	if (rc) return rc;
	P.sweep = sweep; P.nRandomIters = nRandomIters;
	for (int colour = 0; colour < 2; ++colour) {
		if (half >= 0 && half != colour) continue;
		P.colour = colour;
		CK(pm_launch_sweep(P, ctx->tmapValid ? &ctx->tmapRef : nullptr, !ctx->dbg.scalarTaps, geom, ctx->dbg.sweepFourCtas != 0, s));
	}
	return B200MVS_OK;
}
int b200mvs_pm_finalize(b200mvs_ctx* ctx, int width, int height, float keep, const float* plane4, const float* cost,
	float* depth, float* normal, float* conf, void* stream)
{
	if (!ctx || !plane4 || !cost || !depth || !normal || !conf) return B200MVS_ERR_ARG;
	CK(cudaSetDevice(ctx->device));
	CK(pm_launch_finalize(width*height, keep, (const float4*)plane4, cost, nullptr, depth, normal, conf, nullptr,
		stream ? (cudaStream_t)stream : ctx->stream));
	return B200MVS_OK;
}

// ---- SGM --------------------------------------------------------------------------------------
void b200mvs_sgm_default_params(b200mvs_sgm_params* p) { p->P1 = 3; p->P2 = 4; p->P2alpha = 14.f; p->P2beta = 38.f; }

namespace {
// b200mvs_sgm_match_device; known8 != NULL: the pixel-map statistics of sgm_launch_maxdisp, already read back by the caller
int sgm_match(b200mvs_ctx* ctx, const float* leftGray, const uint8_t* leftBGR, const float* rightGray,
	int width, int height, const b200mvs_sgm_pixel* pixels, uint64_t numCosts, const b200mvs_sgm_params* prm,
	int stages, uint8_t* costs, uint16_t* accums, int16_t* disparity, uint16_t* cost, void* stream, b200mvs_stats* stats, const int* known8)
{
	if (!ctx) return B200MVS_ERR_ARG;
	if (!leftGray || !leftBGR || !rightGray || !pixels || width <= 6 || height <= 6 || numCosts == 0)
		return fail(ctx, B200MVS_ERR_ARG, "sgm: null image/pixel map or image too small");
	if ((stages & 4) && (!disparity || !cost))
		return fail(ctx, B200MVS_ERR_ARG, "sgm: null output map");
	b200mvs_sgm_params def; b200mvs_sgm_default_params(&def);
	if (!prm) prm = &def;
	CK(cudaSetDevice(ctx->device));
	cudaStream_t s = stream ? (cudaStream_t)stream : ctx->stream;
	static_assert(sizeof(b200mvs_sgm_pixel) == sizeof(SGMPixel), "pixel record layout");
	SGMParams P; memset(&P, 0, sizeof(P));
	P.lgray = leftGray; P.lbgr = (const uchar3*)leftBGR; P.rgray = rightGray;
	P.w = width; P.h = height; P.vw = width-6; P.vh = height-6;
	P.px = (const SGMPixel*)pixels;
	P.P1 = prm->P1;
	int minP2 = 1<<30, maxP2 = 0;
	for (int i = 0; i < 256; ++i) {
		// GenerateP2s (libs/MVS/SemiGlobalMatcher.cpp:518-524)
		P.P2s[i] = (uint16_t)(int)std::floor(prm->P2*(1.f+prm->P2alpha*std::exp(-float(i)*float(i)/(2.f*prm->P2beta*prm->P2beta)))+.5f);
		minP2 = std::min(minP2, (int)P.P2s[i]); maxP2 = std::max(maxP2, (int)P.P2s[i]);
	}
	if (prm->P1 < 0 || prm->P1 > minP2)
		return fail(ctx, B200MVS_ERR_ARG, "sgm: needs 0 <= P1 <= min(P2s)");
	if (!costs) { CK(ctx->sgCosts.reserve(numCosts)); costs = ctx->sgCosts.as<uint8_t>(); }
	if (!accums) { CK(ctx->sgAccums.reserve(numCosts*sizeof(uint16_t))); accums = ctx->sgAccums.as<uint16_t>(); }
	P.costs = costs; P.accums = accums;
	const auto t0 = std::chrono::steady_clock::now();
	ctx->launches = 0;
	int st8[8] = {0, 0, 0, 0, 0, 0, 0, 0}; bool uniform = false, ring = false, front = false;
	const int mode = ctx->dbg.sgmAggregation;
	if (stats) CK(cudaEventRecord(ctx->ev0, s));
	if (stages & 7) {
		// the warp-per-scanline kernel keeps one line of at most sgm_max_disparities() values
		if (known8) memcpy(st8, known8, sizeof(st8));
		else {
			CK(ctx->sgMax.reserve(8*sizeof(int)));
			CK(sgm_launch_maxdisp(P.px, P.vw*P.vh, numCosts, ctx->sgMax.as<int>(), s)); ctx->launches += 2;
			CK(cudaMemcpyAsync(st8, ctx->sgMax.p, 8*sizeof(int), cudaMemcpyDeviceToHost, s));
			CK(cudaStreamSynchronize(s));
		}
		if (st8[7])
			return fail(ctx, B200MVS_ERR_ARG, "sgm: a pixel's slice [idx, idx+dmax-dmin) ends beyond numCosts");
		if (st8[0] > sgm_max_disparities())
			return fail(ctx, B200MVS_ERR_ARG, "sgm: more than 256 disparities per pixel");
		P.maxNumDisp = st8[0];
		// one global range (the non-tSGM branch): packed, shared-memory-free aggregation kernels
		uniform = st8[0] >= 4 && st8[1] == st8[2] && st8[3] == st8[4] && (st8[0] & 3) == 0 && (st8[5] & 3) == 0 && mode != 1;
		// every slice 16-byte aligned: bulk-copy ring kernel (one launch per direction)
		ring = uniform && (st8[0] & 15) == 0 && st8[5] == 0 && !((uintptr_t)P.costs & 15) && !((uintptr_t)P.accums & 15) && mode != 2;
		// dense volume of a supported width: wave-front kernel (fused directions) — the default
		// (its step carries P2 + the previous line's minimum in 16 bits: P2 <= 16000; sums of eight paths overflow far earlier)
		front = ring && !st8[6] && sgm_front_supports(st8[0]) && maxP2 <= 16000 && (mode == 0 || mode == 4);
		if (mode == 4 && !front)
			return fail(ctx, B200MVS_ERR_ARG, "sgm: the wave-front kernel needs a dense volume with one range of 64, 128 or 256 disparities");
	}
	if (stages & 1) {
		// dense volume with one range of 64 / 128 disparities: the banded-GEMM cost kernel on the tensor cores (sgm_cost_tc.cu)
		const bool dense = uniform && (st8[0] & 15) == 0 && !st8[6] && !((uintptr_t)P.costs & 15);
		const bool tc = dense && sgm_cost_tc_supports(st8[0]) && ctx->dbg.sgmCost != 1;   // auto: the tensor-core kernel where it applies
		if (ctx->dbg.sgmCost == 2 && !tc)
			return fail(ctx, B200MVS_ERR_ARG, "sgm: the tensor-core cost kernel needs a dense volume with one range of 64, 128, 192 or 256 disparities");
		if (tc) { CK(sgm_cost_tc_launch(P, st8[1], st8[0], s)); ctx->launches += (st8[0]+127)/128; }
		else { CK(sgm_launch_cost(P, s)); ++ctx->launches; }
	}
	bool twoVolumes = false;   // the wave-front passes ran side by side: accums + ctx->sgAccums2 is the sum
	bool eightVolumes = false; // ragged ranges: one volume per direction, accums + the seven of ctx->sgAccums2
	if ((stages & 2) && front) {
		const int rc = sgm_aggregate_fronts(ctx, P, st8[0], s, twoVolumes);
		if (rc) return rc;
		if (twoVolumes && !(stages & 4)) { CK(sgm_launch_wta_uniform(P, ctx->sgAccums2.as<uint16_t>(), st8[1], st8[0], nullptr, nullptr, s)); ++ctx->launches; }
	} else
	if ((stages & 2) && !uniform && numCosts <= (1ull<<28)) {
		// ragged (tSGM) ranges: a direction has only 1000-3000 scanlines, one warp each — far too few to fill the GPU.  The eight
		// directions run side by side on eight streams, each STORING its path costs into a volume of its own (no memset, no
		// read-modify-write, no races); the winner-takes-all kernel adds the volumes.
		eightVolumes = true;
		CK(ctx->sgAccums2.reserve((size_t)7*numCosts*sizeof(uint16_t)));
		if (!ctx->sgSide[0]) {
			for (int i = 0; i < 7; ++i) { CK(cudaStreamCreateWithFlags(&ctx->sgSide[i], cudaStreamNonBlocking)); CK(cudaEventCreateWithFlags(&ctx->sgJoin[i], cudaEventDisableTiming)); }
			CK(cudaEventCreateWithFlags(&ctx->sgFork, cudaEventDisableTiming));
		}
		CK(cudaEventRecord(ctx->sgFork, s));
		for (int dir = 0; dir < 8; ++dir) {
			SGMParams Pd = P;
			cudaStream_t sd = s;
			if (dir > 0) {
				Pd.accums = ctx->sgAccums2.as<uint16_t>() + (size_t)(dir-1)*numCosts;
				sd = ctx->sgSide[dir-1];
				CK(cudaStreamWaitEvent(sd, ctx->sgFork, 0));
			}
			CK(sgm_launch_aggregate(Pd, dir, true, sd));
			++ctx->launches;
			if (dir > 0) { CK(cudaEventRecord(ctx->sgJoin[dir-1], sd)); CK(cudaStreamWaitEvent(s, ctx->sgJoin[dir-1], 0)); }
		}
		if (!(stages & 4)) { CK(sgm_launch_wta(P, 8, numCosts, ctx->sgAccums2.as<uint16_t>(), nullptr, nullptr, s)); ++ctx->launches; }
	} else
	if (stages & 2) {
		CK(cudaMemsetAsync(accums, 0, numCosts*sizeof(uint16_t), s));
		for (int dir = 0; dir < 8; ++dir) {
			if (uniform) CK(sgm_launch_aggregate_uniform(P, dir, st8[1], st8[0], ring, s));
			else CK(sgm_launch_aggregate(P, dir, false, s));
			++ctx->launches;
		}
	}
	if (stages & 2) { ctx->sgLastPx = (accums == ctx->sgAccums.as<uint16_t>()) ? (const void*)pixels : nullptr; ctx->sgLastNum = numCosts; ctx->sgFrontRan = front; }
	if (stages & 4) {
		const bool denseWta = uniform && (st8[0] & 15) == 0 && !st8[6] && !((uintptr_t)P.accums & 15);
		if (denseWta) CK(sgm_launch_wta_uniform(P, twoVolumes ? ctx->sgAccums2.as<uint16_t>() : nullptr, st8[1], st8[0], disparity, cost, s));
		else CK(sgm_launch_wta(P, eightVolumes ? 8 : 1, numCosts, eightVolumes ? ctx->sgAccums2.as<uint16_t>() : nullptr, disparity, cost, s));
		++ctx->launches;
	}
	if (stats) {
		CK(cudaEventRecord(ctx->ev1, s));
		CK(cudaStreamSynchronize(s));
		float ms = 0; CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
		memset(stats, 0, sizeof(*stats));
		stats->ms_device = ms;
		stats->ms_total = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now()-t0).count();
		stats->kernel_launches = ctx->launches; stats->levels = 1;
		if ((stages & 2) && front) {
			// the wave-front kernel flags a dependency wait that timed out (never in a correct schedule): the stream is idle here
			int err = 0;
			CK(cudaMemcpy(&err, ctx->sgFrontCtl.as<int>()+1, sizeof(int), cudaMemcpyDeviceToHost));
			if (err) return fail(ctx, B200MVS_ERR_CUDA, "sgm: the wave-front aggregation timed out waiting for a predecessor");
		}
	}
	return B200MVS_OK;
}
} // namespace

int b200mvs_sgm_match_device(b200mvs_ctx* ctx, const float* leftGray, const uint8_t* leftBGR, const float* rightGray,
	int width, int height, const b200mvs_sgm_pixel* pixels, uint64_t numCosts, const b200mvs_sgm_params* prm,
	int stages, uint8_t* costs, uint16_t* accums, int16_t* disparity, uint16_t* cost, void* stream, b200mvs_stats* stats)
{
	return sgm_match(ctx, leftGray, leftBGR, rightGray, width, height, pixels, numCosts, prm, stages, costs, accums, disparity, cost,
		stream, stats, nullptr);
}

int b200mvs_sgm_match(b200mvs_ctx* ctx, const float* leftGray, const uint8_t* leftBGR, const float* rightGray,
	int width, int height, const b200mvs_sgm_pixel* pixels, uint64_t numCosts, const b200mvs_sgm_params* prm,
	int16_t* disparity, uint16_t* cost, b200mvs_stats* stats)
{
	if (!ctx) return B200MVS_ERR_ARG;
	if (!leftGray || !leftBGR || !rightGray || !pixels || !disparity || !cost || width <= 6 || height <= 6)
		return fail(ctx, B200MVS_ERR_ARG, "sgm: null pointer or image too small");
	CK(cudaSetDevice(ctx->device));
	cudaStream_t s = ctx->stream;
	const auto t0 = std::chrono::steady_clock::now();
	const size_t n = (size_t)width*height, nv = (size_t)(width-6)*(height-6);
	CK(ctx->sgL.reserve(n*4)); CK(ctx->sgR.reserve(n*4)); CK(ctx->sgC.reserve(n*3)); CK(ctx->sgPx.reserve(nv*sizeof(SGMPixel)));
	CK(ctx->sgDisp.reserve(nv*2)); CK(ctx->sgCost.reserve(nv*2));
	CK(cudaMemcpyAsync(ctx->sgL.p, leftGray, n*4, cudaMemcpyHostToDevice, s));
	CK(cudaMemcpyAsync(ctx->sgR.p, rightGray, n*4, cudaMemcpyHostToDevice, s));
	CK(cudaMemcpyAsync(ctx->sgC.p, leftBGR, n*3, cudaMemcpyHostToDevice, s));
	CK(cudaMemcpyAsync(ctx->sgPx.p, pixels, nv*sizeof(SGMPixel), cudaMemcpyHostToDevice, s));
	b200mvs_stats st;
	int rc = b200mvs_sgm_match_device(ctx, ctx->sgL.as<float>(), ctx->sgC.as<uint8_t>(), ctx->sgR.as<float>(), width, height,
		(const b200mvs_sgm_pixel*)ctx->sgPx.p, numCosts, prm, 7, nullptr, nullptr, ctx->sgDisp.as<int16_t>(), ctx->sgCost.as<uint16_t>(), s, &st);
	if (rc) return rc;
	CK(cudaMemcpyAsync(disparity, ctx->sgDisp.p, nv*2, cudaMemcpyDeviceToHost, s));
	CK(cudaMemcpyAsync(cost, ctx->sgCost.p, nv*2, cudaMemcpyDeviceToHost, s));
	CK(cudaStreamSynchronize(s));
	if (stats) {
		*stats = st;
		stats->bytes_h2d = n*11+nv*sizeof(SGMPixel); stats->bytes_d2h = nv*4;
		stats->ms_total = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now()-t0).count();
	}
	return B200MVS_OK;
}

int b200mvs_sgm_cross_check_device(b200mvs_ctx* ctx, int16_t* l2r, const int16_t* r2l, int width, int height, int thCross, void* stream) {
	if (!ctx || !l2r || !r2l || width <= 0 || height <= 0 || thCross < 0) return B200MVS_ERR_ARG;
	CK(cudaSetDevice(ctx->device));
	CK(sgm_launch_cross_check(l2r, r2l, width, height, thCross, stream ? (cudaStream_t)stream : ctx->stream));
	return B200MVS_OK;
}

int b200mvs_sgm_refine_device(b200mvs_ctx* ctx, const b200mvs_sgm_pixel* pixels, const uint16_t* accums, int16_t* disparity,
	int nPixels, int subpixelSteps, void* stream)
{
	if (!ctx || !pixels || !disparity || nPixels <= 0) return B200MVS_ERR_ARG;
	if (!accums) {
		// the accumulated costs of the last match on this context: only valid for the pixel map they were computed for
		accums = ctx->sgAccums.as<uint16_t>();
		if (!accums || ctx->sgLastPx != (const void*)pixels)
			return fail(ctx, B200MVS_ERR_ARG, "sgm refine: no accumulated costs of a match with this pixel map on the context");
	}
	if (subpixelSteps <= 1) return B200MVS_OK;
	CK(cudaSetDevice(ctx->device));
	CK(sgm_launch_refine((const SGMPixel*)pixels, accums, disparity, nPixels, subpixelSteps, stream ? (cudaStream_t)stream : ctx->stream));
	return B200MVS_OK;
}

// ---- coarse-to-fine (tSGM) matching of a rectified pair: the level loop of SemiGlobalMatcher::Match(scene, ...) ----
// (libs/MVS/SemiGlobalMatcher.cpp:584-718; the per-level steps are in sgm_tsgm.cu, the matches are sgm_match)
namespace {

inline int cv_round(double v) { return (int)std::nearbyint(v); }   // cv::saturate_cast<int>(double)

// computeMaxResolution (libs/Common/Types.inl:2459-2477) with level = 8, scale = 1/max(2, 2^level) (SemiGlobalMatcher.cpp:584-589);
// the seed is the valid region of computeResize(coarsest level, 0.5) (:620-624)
void tsgm_levels(int width, int height, int minResolution, int& nLevels, int& seedWidth, int& seedHeight) {
	const unsigned imageSize = (unsigned)std::max(width, height);
	unsigned level = 8;
	if ((imageSize >> level) < (unsigned)minResolution) {
		level = 0;
		while ((imageSize >> (level+1)) >= (unsigned)minResolution)
			++level;
	}
	const int L = (int)std::max(1u, level);
	nLevels = L+1;
	const int cw = cv_round(width/(double)(1 << L)), ch = cv_round(height/(double)(1 << L));
	seedWidth = cv_round(cw*0.5)-6; seedHeight = cv_round(ch*0.5)-6;
}

// Disparity2RangeMap's layout needs the fine valid region to reach past 2 x the coarse map plus the 3-pixel offset
inline bool range_sizes_ok(int dw, int dh, int mw, int mh) { return dw > 0 && dh > 0 && mw >= 2*dw+4 && mh >= 2*dh+2 && mw < 32768; }

// Disparity2RangeMap into `pixels`; with st8 != NULL also the statistics the match needs (sgm_launch_maxdisp).  One read-back:
// the volume of the following match is sized from it.
int ts_range_map(b200mvs_ctx* ctx, const int16_t* D, int dw, int dh, const uint8_t* M, int mw, int mh, int minND, int minNDI,
	void* pixels, uint64_t& numCosts, int& maxNumDisp, int* st8, cudaStream_t s)
{
	CK(ctx->tsRange.reserve((size_t)dw*dh*4));
	CK(ctx->tsScratch.reserve(ts_range_scratch_bytes(mw, mh)));
	CK(ctx->tsStat.reserve(64));
	unsigned long long* stat = ctx->tsStat.as<unsigned long long>();
	CK(ts_launch_range_map(D, dw, dh, M, mw, mh, minND, minNDI, ctx->tsRange.as<uint32_t>(), ctx->tsScratch.p, pixels, stat, s));
	ctx->launches += 5;
	if (st8) { CK(sgm_launch_maxdisp((const SGMPixel*)pixels, mw*mh, ~0ull, (int*)(stat+2), s)); ctx->launches += 2; }
	unsigned long long host[6];
	CK(cudaMemcpyAsync(host, stat, st8 ? 48 : 16, cudaMemcpyDeviceToHost, s));
	CK(cudaStreamSynchronize(s));
	numCosts = host[0];
	maxNumDisp = (int)(uint32_t)host[1];
	if (st8) memcpy(st8, host+2, 8*sizeof(int));
	return B200MVS_OK;
}

// the wave-front aggregation flags a dependency wait that timed out (never in a correct schedule)
int ts_check_front(b200mvs_ctx* ctx, cudaStream_t s) {
	if (!ctx->sgFrontRan) return B200MVS_OK;
	int err = 0;
	CK(cudaMemcpyAsync(&err, ctx->sgFrontCtl.as<int>()+1, sizeof(int), cudaMemcpyDeviceToHost, s));
	CK(cudaStreamSynchronize(s));
	if (err) return fail(ctx, B200MVS_ERR_CUDA, "sgm: the wave-front aggregation timed out waiting for a predecessor");
	return B200MVS_OK;
}

} // namespace

int b200mvs_sgm_tsgm_levels(int width, int height, int minResolution, int* nLevels, int* seedWidth, int* seedHeight) {
	if (!nLevels || !seedWidth || !seedHeight || width <= 0 || height <= 0 || minResolution <= 0) return B200MVS_ERR_ARG;
	tsgm_levels(width, height, minResolution, *nLevels, *seedWidth, *seedHeight);
	return B200MVS_OK;
}

int b200mvs_sgm_match_tsgm_device(b200mvs_ctx* ctx, const float* leftGray, const uint8_t* leftBGR, const float* rightGray, const uint8_t* rightBGR,
	int width, int height, const uint8_t* leftMask, const uint8_t* rightMask, int maskWidth, int maskHeight,
	const int16_t* seed, int seedWidth, int seedHeight, int minResolution, int nSpeckleSize, int subpixelSteps,
	const b200mvs_sgm_params* prm, int16_t* disparity, uint16_t* cost, void* stream, b200mvs_stats* stats)
{
	if (!ctx) return B200MVS_ERR_ARG;
	if (!leftGray || !leftBGR || !rightGray || !rightBGR || !disparity || !cost || width <= 6 || height <= 6 || width >= 32768 || height >= 32768)
		return fail(ctx, B200MVS_ERR_ARG, "sgm tsgm: null image or output, or image size out of range");
	if (minResolution <= 0 || nSpeckleSize < 0 || subpixelSteps < 1)
		return fail(ctx, B200MVS_ERR_ARG, "sgm tsgm: needs minResolution > 0, nSpeckleSize >= 0, subpixelSteps >= 1");
	if ((leftMask || rightMask) && (maskWidth != width || maskHeight != height))
		return fail(ctx, B200MVS_ERR_ARG, "sgm tsgm: the masks must have the size of the images");
	int nLevels, sw, sh;
	tsgm_levels(width, height, minResolution, nLevels, sw, sh);
	if (seed && (seedWidth != sw || seedHeight != sh))
		return fail(ctx, B200MVS_ERR_ARG, "sgm tsgm: the seed must be computeResize(coarsest level, 0.5) minus 6 (b200mvs_sgm_tsgm_levels)");
	{
		int pw = sw, ph = sh;
		for (int level = 0; level < nLevels; ++level) {
			const int f = 1 << (nLevels-1-level);
			const int vw = cv_round(width/(double)f)-6, vh = cv_round(height/(double)f)-6;
			if (!range_sizes_ok(pw, ph, vw, vh))
				return fail(ctx, B200MVS_ERR_ARG, "sgm tsgm: image too small for this minResolution");
			pw = vw; ph = vh;
		}
	}
	b200mvs_sgm_params def; b200mvs_sgm_default_params(&def);
	if (!prm) prm = &def;
	CK(cudaSetDevice(ctx->device));
	cudaStream_t s = stream ? (cudaStream_t)stream : ctx->stream;
	const auto t0 = std::chrono::steady_clock::now();
	int launches = 0;
	if (stats) CK(cudaEventRecord(ctx->ev0, s));
	const size_t nv = (size_t)(width-6)*(height-6), n = (size_t)width*height;
	// level images of every level below full resolution fit the half-resolution level
	const size_t nHalf = (size_t)(cv_round(width*0.5)+1)*(cv_round(height*0.5)+1);
	CK(ctx->tsLG.reserve(nHalf*4)); CK(ctx->tsRG.reserve(nHalf*4)); CK(ctx->tsLC.reserve(nHalf*3)); CK(ctx->tsRC.reserve(nHalf*3));
	CK(ctx->tsDisp.reserve(4*nv*2)); CK(ctx->tsMask.reserve(4*nv+n)); CK(ctx->tsLab.reserve(2*nv*4));
	CK(ctx->tsCost.reserve(nv*2)); CK(ctx->tsPx.reserve(nv*sizeof(SGMPixel)));
	int16_t* dbuf[2] = {ctx->tsDisp.as<int16_t>(), ctx->tsDisp.as<int16_t>()+nv};
	int16_t* rFlip = ctx->tsDisp.as<int16_t>()+2*nv;
	int16_t* rD = ctx->tsDisp.as<int16_t>()+3*nv;
	uint8_t* mbuf[2][2] = {{ctx->tsMask.as<uint8_t>(), ctx->tsMask.as<uint8_t>()+nv}, {ctx->tsMask.as<uint8_t>()+2*nv, ctx->tsMask.as<uint8_t>()+3*nv}};
	uint8_t* maskTmp = ctx->tsMask.as<uint8_t>()+4*nv;
	int* lab = ctx->tsLab.as<int>();
	void* px = ctx->tsPx.p;
	const int16_t* lPrev = seed;
	if (!seed) { CK(ts_launch_fill_i16(dbuf[0], (size_t)sw*sh, 32767, s)); ++launches; lPrev = dbuf[0]; }
	int pw = sw, ph = sh, cur = 0;   // size of the previous level's maps, mask ping-pong slot
	for (int level = 0; level < nLevels; ++level) {
		const int f = 1 << (nLevels-1-level);
		const bool first = level == 0, last = level+1 == nLevels;
		// ViewData::GetImage(scale) (SemiGlobalMatcher.h:127-142)
		int lw = width, lh = height;
		const float *LG = leftGray, *RG = rightGray; const uint8_t *LC = leftBGR, *RC = rightBGR;
		if (f > 1) {
			lw = cv_round(width/(double)f); lh = cv_round(height/(double)f);
			CK(rs_launch_area(leftGray, width, height, width, ctx->tsLG.as<float>(), lw, lh, f, f, s));
			CK(rs_launch_area(rightGray, width, height, width, ctx->tsRG.as<float>(), lw, lh, f, f, s));
			CK(ts_launch_resize_area_u8(leftBGR, width, height, 3, f, ctx->tsLC.as<uint8_t>(), lw, lh, s));
			CK(ts_launch_resize_area_u8(rightBGR, width, height, 3, f, ctx->tsRC.as<uint8_t>(), lw, lh, s));
			launches += 4;
			LG = ctx->tsLG.as<float>(); RG = ctx->tsRG.as<float>(); LC = ctx->tsLC.as<uint8_t>(); RC = ctx->tsRC.as<uint8_t>();
		}
		const int vw = lw-6, vh = lh-6;
		const size_t nl = (size_t)vw*vh;
		uint8_t* lM = mbuf[cur^1][0];
		uint8_t* rM = mbuf[cur^1][1];
		for (int m = 0; m < 2; ++m) {
			uint8_t* dst = m == 0 ? lM : rM;
			const uint8_t* src = m == 0 ? leftMask : rightMask;
			if (!first) { CK(ts_launch_upscale_mask(mbuf[cur][m], pw, ph, dst, vw, vh, s)); ++launches; }
			else if (!src) CK(cudaMemsetAsync(dst, 255, nl, s));
			else {
				// NEAREST to the level size, then the valid ROI (:626-631)
				CK(rs_launch_nearest_u8(src, width, height, width, maskTmp, lw, lh, s)); ++launches;
				CK(cudaMemcpy2DAsync(dst, vw, maskTmp+3*lw+3, lw, vw, vh, cudaMemcpyDeviceToDevice, s));
			}
		}
		cur ^= 1;
		const int minND = first ? 11 : 5, minNDI = first ? 33 : 7;
		int16_t* lCur = last ? disparity : (lPrev == dbuf[0] ? dbuf[1] : dbuf[0]);
		uint16_t* lCost = last ? cost : ctx->tsCost.as<uint16_t>();
		int st8[8]; uint64_t numCosts; int maxND; int rc;
		auto match = [&](const float* a, const uint8_t* ac, const float* b, int16_t* d, uint16_t* c) -> int {
			if (numCosts == 0) {
				// every pixel masked out: the winner-takes-all of the reference leaves NO_DISP / NO_ACCUMCOST
				CK(ts_launch_fill_i16(d, nl, 32767, s)); ++launches;
				CK(cudaMemsetAsync(c, 0xFF, nl*2, s));
				return B200MVS_OK;
			}
			const int r = sgm_match(ctx, a, ac, b, lw, lh, (const b200mvs_sgm_pixel*)px, numCosts, prm, 7, nullptr, nullptr, d, c, s, nullptr, st8);
			launches += ctx->launches;
			return r ? r : ts_check_front(ctx, s);
		};
		// right -> left: FlipDirection, Disparity2RangeMap, Match(right, left) (:641-642, 672)
		CK(ts_launch_flip(lPrev, rFlip, pw, ph, (uint32_t*)lab, s)); launches += 2;
		ctx->launches = 0;
		if ((rc = ts_range_map(ctx, rFlip, pw, ph, rM, vw, vh, minND, minNDI, px, numCosts, maxND, st8, s))) return rc;
		launches += ctx->launches;
		if ((rc = match(RG, RC, LG, rD, ctx->tsCost.as<uint16_t>()))) return rc;
		// left -> right (:675-685)
		ctx->launches = 0;
		if ((rc = ts_range_map(ctx, lPrev, pw, ph, lM, vw, vh, minND, minNDI, px, numCosts, maxND, st8, s))) return rc;
		launches += ctx->launches;
		if ((rc = match(LG, LC, RG, lCur, lCost))) return rc;
		if (first) {
			// :698-706; the second cross-check reads the already-checked left map
			CK(sgm_launch_cross_check(lCur, rD, vw, vh, 1, s));
			CK(sgm_launch_cross_check(rD, lCur, vw, vh, 1, s));
			CK(ts_launch_filter_speckles(lCur, vw, vh, 32767, nSpeckleSize, 5, lab, lab+nv, s));
			CK(ts_launch_filter_speckles(rD, vw, vh, 32767, nSpeckleSize, 5, lab, lab+nv, s));
			CK(ts_launch_extract_mask(lCur, lM, vw, vh, 3, s));
			CK(ts_launch_extract_mask(rD, rM, vw, vh, 3, s));
			launches += 4 + 2*ts_filter_speckles_launches(vw, vh);
		} else {
			CK(sgm_launch_cross_check(lCur, rD, vw, vh, 1, s)); ++launches;
		}
		lPrev = lCur; pw = vw; ph = vh;
		if (last && numCosts > 0 && subpixelSteps > 1) {
			// RefineDisparityMap with the pixel map and the accumulated costs of this last left match (:718)
			CK(sgm_launch_refine((const SGMPixel*)px, ctx->sgAccums.as<uint16_t>(), disparity, (int)nl, subpixelSteps, s)); ++launches;
		}
	}
	ctx->sgLastPx = nullptr;
	ctx->launches = launches;
	if (stats) {
		CK(cudaEventRecord(ctx->ev1, s));
		CK(cudaStreamSynchronize(s));
		float ms = 0; CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
		memset(stats, 0, sizeof(*stats));
		stats->ms_device = ms;
		stats->ms_total = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now()-t0).count();
		stats->kernel_launches = launches; stats->levels = nLevels;
	}
	return B200MVS_OK;
}

int b200mvs_sgm_match_tsgm(b200mvs_ctx* ctx, const float* leftGray, const uint8_t* leftBGR, const float* rightGray, const uint8_t* rightBGR,
	int width, int height, const uint8_t* leftMask, const uint8_t* rightMask, int maskWidth, int maskHeight,
	const int16_t* seed, int seedWidth, int seedHeight, int minResolution, int nSpeckleSize, int subpixelSteps,
	const b200mvs_sgm_params* prm, int16_t* disparity, uint16_t* cost, b200mvs_stats* stats)
{
	if (!ctx) return B200MVS_ERR_ARG;
	if (!leftGray || !leftBGR || !rightGray || !rightBGR || !disparity || !cost || width <= 6 || height <= 6 || width >= 32768 || height >= 32768)
		return fail(ctx, B200MVS_ERR_ARG, "sgm tsgm: null image or output, or image size out of range");
	if ((leftMask || rightMask) && (maskWidth != width || maskHeight != height))
		return fail(ctx, B200MVS_ERR_ARG, "sgm tsgm: the masks must have the size of the images");
	int nLevels, sw, sh;
	if (minResolution <= 0) return fail(ctx, B200MVS_ERR_ARG, "sgm tsgm: needs minResolution > 0");
	tsgm_levels(width, height, minResolution, nLevels, sw, sh);
	if (seed && (seedWidth != sw || seedHeight != sh))
		return fail(ctx, B200MVS_ERR_ARG, "sgm tsgm: the seed must be computeResize(coarsest level, 0.5) minus 6 (b200mvs_sgm_tsgm_levels)");
	CK(cudaSetDevice(ctx->device));
	cudaStream_t s = ctx->stream;
	const auto t0 = std::chrono::steady_clock::now();
	const size_t n = (size_t)width*height, nv = (size_t)(width-6)*(height-6), ns = seed ? (size_t)sw*sh : 0;
	CK(ctx->sgL.reserve(n*4)); CK(ctx->sgR.reserve(n*4)); CK(ctx->sgC.reserve(n*6+2*n+ns*2));
	CK(ctx->sgDisp.reserve(nv*2)); CK(ctx->sgCost.reserve(nv*2));
	uint8_t* lc = ctx->sgC.as<uint8_t>(); uint8_t* rc = lc+3*n; uint8_t* lm = rc+3*n; uint8_t* rm = lm+n;
	int16_t* sd = (int16_t*)(rm+n);
	CK(cudaMemcpyAsync(ctx->sgL.p, leftGray, n*4, cudaMemcpyHostToDevice, s));
	CK(cudaMemcpyAsync(ctx->sgR.p, rightGray, n*4, cudaMemcpyHostToDevice, s));
	CK(cudaMemcpyAsync(lc, leftBGR, n*3, cudaMemcpyHostToDevice, s));
	CK(cudaMemcpyAsync(rc, rightBGR, n*3, cudaMemcpyHostToDevice, s));
	if (leftMask) CK(cudaMemcpyAsync(lm, leftMask, n, cudaMemcpyHostToDevice, s));
	if (rightMask) CK(cudaMemcpyAsync(rm, rightMask, n, cudaMemcpyHostToDevice, s));
	if (seed) CK(cudaMemcpyAsync(sd, seed, ns*2, cudaMemcpyHostToDevice, s));
	b200mvs_stats st;
	int r = b200mvs_sgm_match_tsgm_device(ctx, ctx->sgL.as<float>(), lc, ctx->sgR.as<float>(), rc, width, height,
		leftMask ? lm : nullptr, rightMask ? rm : nullptr, maskWidth, maskHeight, seed ? sd : nullptr, seedWidth, seedHeight,
		minResolution, nSpeckleSize, subpixelSteps, prm, ctx->sgDisp.as<int16_t>(), ctx->sgCost.as<uint16_t>(), s, &st);
	if (r) return r;
	CK(cudaMemcpyAsync(disparity, ctx->sgDisp.p, nv*2, cudaMemcpyDeviceToHost, s));
	CK(cudaMemcpyAsync(cost, ctx->sgCost.p, nv*2, cudaMemcpyDeviceToHost, s));
	CK(cudaStreamSynchronize(s));
	if (stats) {
		*stats = st;
		stats->bytes_h2d = n*14 + (leftMask ? n : 0) + (rightMask ? n : 0) + ns*2; stats->bytes_d2h = nv*4;
		stats->ms_total = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now()-t0).count();
	}
	return B200MVS_OK;
}

int b200mvs_sgm_range_map_device(b200mvs_ctx* ctx, const int16_t* disparity, int width, int height, const uint8_t* mask, int maskWidth, int maskHeight,
	int minNumDisp, int minNumDispInvalid, b200mvs_sgm_pixel* pixels, uint64_t* numCosts, int* maxNumDisp, void* stream)
{
	if (!ctx) return B200MVS_ERR_ARG;
	if (!disparity || !mask || !pixels || !range_sizes_ok(width, height, maskWidth, maskHeight))
		return fail(ctx, B200MVS_ERR_ARG, "sgm range map: null pointer, or the mask is not at least (2w+4) x (2h+2)");
	CK(cudaSetDevice(ctx->device));
	uint64_t nc; int mx;
	ctx->launches = 0;
	const int rc = ts_range_map(ctx, disparity, width, height, mask, maskWidth, maskHeight, minNumDisp, minNumDispInvalid, pixels, nc, mx,
		nullptr, stream ? (cudaStream_t)stream : ctx->stream);
	if (rc) return rc;
	if (numCosts) *numCosts = nc;
	if (maxNumDisp) *maxNumDisp = mx;
	return B200MVS_OK;
}

int b200mvs_sgm_flip_direction_device(b200mvs_ctx* ctx, const int16_t* l2r, int16_t* r2l, int width, int height, void* stream) {
	if (!ctx) return B200MVS_ERR_ARG;
	if (!l2r || !r2l || width <= 0 || height <= 0 || width >= 32768) return fail(ctx, B200MVS_ERR_ARG, "sgm flip: null pointer or size out of range");
	CK(cudaSetDevice(ctx->device));
	CK(ctx->tsLab.reserve((size_t)width*height*4));
	CK(ts_launch_flip(l2r, r2l, width, height, ctx->tsLab.as<uint32_t>(), stream ? (cudaStream_t)stream : ctx->stream));
	return B200MVS_OK;
}

int b200mvs_sgm_filter_speckles_device(b200mvs_ctx* ctx, int16_t* disparity, int width, int height, int newVal, int maxSpeckleSize, int maxDiff, void* stream) {
	if (!ctx) return B200MVS_ERR_ARG;
	if (!disparity || width <= 0 || height <= 0 || (size_t)width*height >= (1u << 31) || maxDiff < 0)
		return fail(ctx, B200MVS_ERR_ARG, "sgm filter speckles: null map, size out of range or maxDiff < 0");
	CK(cudaSetDevice(ctx->device));
	const size_t n = (size_t)width*height;
	CK(ctx->tsLab.reserve(n*8));
	CK(ts_launch_filter_speckles(disparity, width, height, newVal, maxSpeckleSize, maxDiff, ctx->tsLab.as<int>(), ctx->tsLab.as<int>()+n,
		stream ? (cudaStream_t)stream : ctx->stream));
	return B200MVS_OK;
}

int b200mvs_sgm_extract_mask_device(b200mvs_ctx* ctx, const int16_t* disparity, uint8_t* mask, int width, int height, int thValid, void* stream) {
	if (!ctx) return B200MVS_ERR_ARG;
	if (!disparity || !mask || width <= 0 || height <= 0) return fail(ctx, B200MVS_ERR_ARG, "sgm extract mask: null pointer or empty map");
	CK(cudaSetDevice(ctx->device));
	CK(ts_launch_extract_mask(disparity, mask, width, height, thValid, stream ? (cudaStream_t)stream : ctx->stream));
	return B200MVS_OK;
}

int b200mvs_sgm_upscale_mask_device(b200mvs_ctx* ctx, const uint8_t* mask, int width, int height, uint8_t* mask2x, int width2, int height2, void* stream) {
	if (!ctx) return B200MVS_ERR_ARG;
	if (!mask || !mask2x || width <= 0 || height <= 0 || width2 <= 0 || height2 <= 0) return fail(ctx, B200MVS_ERR_ARG, "sgm upscale mask: null pointer or empty map");
	CK(cudaSetDevice(ctx->device));
	CK(ts_launch_upscale_mask(mask, width, height, mask2x, width2, height2, stream ? (cudaStream_t)stream : ctx->stream));
	return B200MVS_OK;
}

int b200mvs_resize_area_bgr8_device(b200mvs_ctx* ctx, const uint8_t* image, int width, int height, int factor, uint8_t* resized, void* stream) {
	if (!ctx) return B200MVS_ERR_ARG;
	if (!image || !resized || width <= 0 || height <= 0 || factor < 2) return fail(ctx, B200MVS_ERR_ARG, "resize area bgr8: null pointer, empty image or factor < 2");
	const int dw = cv_round(width/(double)factor), dh = cv_round(height/(double)factor);
	if (dw <= 0 || dh <= 0) return fail(ctx, B200MVS_ERR_ARG, "resize area bgr8: resized image is empty");
	CK(cudaSetDevice(ctx->device));
	CK(ts_launch_resize_area_u8(image, width, height, 3, factor, resized, dw, dh, stream ? (cudaStream_t)stream : ctx->stream));
	return B200MVS_OK;
}

// ---- depth-map post-processing (SceneDensify.cpp:810-1299) ----

void b200mvs_filter_default_params(b200mvs_filter_params* p) {
	p->nMinViews = 2; p->nMinViewsAdjust = 1; p->fDepthDiffThreshold = 0.01f; p->bAdjust = 1;
}

static void flt_view(const b200mvs_dmap& m, const float* depth, const float* conf, FltView& v) {
	v.depth = depth; v.conf = conf; v.w = m.width; v.h = m.height;
	v.fx = m.K[0]; v.fy = m.K[4]; v.cx = m.K[2]; v.cy = m.K[5];
	memcpy(v.R, m.R, sizeof(v.R)); memcpy(v.C, m.C, sizeof(v.C));
}

static int flt_check(b200mvs_ctx* ctx, const b200mvs_dmap* ref, const b200mvs_dmap* nbrs, int nNbrs, const b200mvs_filter_params* prm,
	const float* outDepth, const float* outConf)
{
	if (!ctx) return B200MVS_ERR_ARG;
	if (!ref || !prm || !outDepth || !outConf || nNbrs < 0 || (nNbrs > 0 && !nbrs))
		return fail(ctx, B200MVS_ERR_ARG, "filter: null pointer");
	if (nNbrs > B200MVS_MAX_FILTER_VIEWS) return fail(ctx, B200MVS_ERR_ARG, "filter: too many neighbour depth-maps");
	if (!ref->depth || !ref->conf || ref->width <= 0 || ref->height <= 0 || (size_t)ref->width*ref->height >= 0xFFFFFFFFull)
		return fail(ctx, B200MVS_ERR_ARG, "filter: invalid reference depth-map");
	if (prm->nMinViews < 1 || prm->nMinViewsAdjust < 0 || !(prm->fDepthDiffThreshold > 0))
		return fail(ctx, B200MVS_ERR_ARG, "filter: invalid parameter block"); // nMinViewsFilter > 0 is asserted by the reference (:1057)
	for (int i = 0; i < nNbrs; ++i) {
		const b200mvs_dmap& m = nbrs[i];
		if (!m.depth || (prm->bAdjust && !m.conf) || m.width <= 0 || m.height <= 0 || (size_t)m.width*m.height >= 0xFFFFFFFFull)
			return fail(ctx, B200MVS_ERR_ARG, "filter: invalid neighbour depth-map");
	}
	return B200MVS_OK;
}

int b200mvs_filter_depth_map_device(b200mvs_ctx* ctx, const b200mvs_dmap* ref, const b200mvs_dmap* nbrs, int nNbrs,
	const b200mvs_filter_params* prm, float dMin, float dMax, float* outDepth, float* outConf,
	float* projDepth, float* projConf, int* filtered, void* stream)
{
	int rc = flt_check(ctx, ref, nbrs, nNbrs, prm, outDepth, outConf);
	if (rc) return rc;
	if (nNbrs < prm->nMinViews || nNbrs < prm->nMinViewsAdjust) { // "can not be filtered" (:1060-1063)
		if (filtered) *filtered = 0;
		return B200MVS_OK;
	}
	CK(cudaSetDevice(ctx->device));
	cudaStream_t s = stream ? (cudaStream_t)stream : ctx->stream;
	const size_t np = (size_t)ref->width*ref->height;
	CK(ctx->fltZ.reserve(np*8*(size_t)nNbrs));
	FltParams P;
	memset(&P, 0, sizeof(P));
	flt_view(*ref, ref->depth, ref->conf, P.ref);
	int maxPix = 0;
	for (int i = 0; i < nNbrs; ++i) {
		flt_view(nbrs[i], nbrs[i].depth, nbrs[i].conf, P.nbr[i]);
		maxPix = std::max(maxPix, nbrs[i].width*nbrs[i].height);
	}
	P.N = nNbrs; P.nMinViews = prm->nMinViews; P.nMinViewsAdjust = prm->nMinViewsAdjust;
	P.thDepthDiff = prm->fDepthDiffThreshold*1.2f; P.thStrict = prm->fDepthDiffThreshold*0.8f;
	P.dMin = dMin; P.dMax = dMax;
	P.zbuf = ctx->fltZ.as<unsigned long long>(); P.outDepth = outDepth; P.outConf = outConf;
	CK(flt_launch_filter(P, maxPix, prm->bAdjust != 0, s));
	ctx->launches = 2;
	if (projDepth) {
		for (int i = 0; i < nNbrs; ++i)
			CK(flt_launch_resolve(P.zbuf+np*i, nbrs[i].conf, np, projDepth+np*i, projConf ? projConf+np*i : nullptr, s));
		ctx->launches += nNbrs;
	}
	if (filtered) *filtered = 1;
	return B200MVS_OK;
}

int b200mvs_filter_depth_map(b200mvs_ctx* ctx, const b200mvs_dmap* ref, const b200mvs_dmap* nbrs, int nNbrs,
	const b200mvs_filter_params* prm, float dMin, float dMax, float* outDepth, float* outConf, int* filtered, b200mvs_stats* stats)
{
	int rc = flt_check(ctx, ref, nbrs, nNbrs, prm, outDepth, outConf);
	if (rc) return rc;
	if (nNbrs < prm->nMinViews || nNbrs < prm->nMinViewsAdjust) { if (filtered) *filtered = 0; return B200MVS_OK; }
	CK(cudaSetDevice(ctx->device));
	cudaStream_t s = ctx->stream;
	const auto t0 = std::chrono::steady_clock::now();
	// stage every map once: [ref depth | ref conf | nbr0 depth | nbr0 conf | ...]
	size_t total = 0;
	for (int i = -1; i < nNbrs; ++i) { const b200mvs_dmap& m = i < 0 ? *ref : nbrs[i]; total += (size_t)m.width*m.height*2; }
	const size_t np = (size_t)ref->width*ref->height;
	CK(ctx->fltIn.reserve(total*4)); CK(ctx->fltOutD.reserve(np*4)); CK(ctx->fltOutC.reserve(np*4));
	std::vector<b200mvs_dmap> dv(nNbrs+1);
	float* p = ctx->fltIn.as<float>();
	uint64_t h2d = 0;
	for (int i = -1; i < nNbrs; ++i) {
		const b200mvs_dmap& m = i < 0 ? *ref : nbrs[i];
		const size_t n = (size_t)m.width*m.height;
		b200mvs_dmap& d = dv[i+1];
		d = m;
		CK(cudaMemcpyAsync(p, m.depth, n*4, cudaMemcpyHostToDevice, s)); d.depth = p; p += n; h2d += n*4;
		d.conf = nullptr;
		if (m.conf) { CK(cudaMemcpyAsync(p, m.conf, n*4, cudaMemcpyHostToDevice, s)); d.conf = p; h2d += n*4; }
		p += n;
	}
	CK(cudaEventRecord(ctx->ev0, s));
	rc = b200mvs_filter_depth_map_device(ctx, &dv[0], dv.data()+1, nNbrs, prm, dMin, dMax, ctx->fltOutD.as<float>(), ctx->fltOutC.as<float>(),
		nullptr, nullptr, filtered, s);
	if (rc) return rc;
	CK(cudaEventRecord(ctx->ev1, s));
	CK(cudaMemcpyAsync(outDepth, ctx->fltOutD.p, np*4, cudaMemcpyDeviceToHost, s));
	CK(cudaMemcpyAsync(outConf, ctx->fltOutC.p, np*4, cudaMemcpyDeviceToHost, s));
	CK(cudaStreamSynchronize(s));
	if (stats) {
		memset(stats, 0, sizeof(*stats));
		float ms = 0; cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
		stats->ms_device = ms; stats->bytes_h2d = h2d; stats->bytes_d2h = np*8; stats->kernel_launches = ctx->launches; stats->levels = 1;
		stats->ms_total = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now()-t0).count();
	}
	return B200MVS_OK;
}

int b200mvs_remove_small_segments_device(b200mvs_ctx* ctx, float* depth, float* normal, float* conf, int width, int height,
	float fDepthDiffThreshold, unsigned nSpeckleSize, void* stream)
{
	if (!ctx) return B200MVS_ERR_ARG;
	if (!depth || width <= 0 || height <= 0 || (size_t)width*height > 0x7FFFFFFFull || !(fDepthDiffThreshold > 0))
		return fail(ctx, B200MVS_ERR_ARG, "remove_small_segments: invalid argument");
	CK(cudaSetDevice(ctx->device));
	const size_t n = (size_t)width*height;
	cudaStream_t s = stream ? (cudaStream_t)stream : ctx->stream;
	const float th = fDepthDiffThreshold*0.7f;
	const int cap = 1<<18;   // one-way edges kept (a 1080p map has tens); beyond it the call fails loudly
	CK(ctx->ppA.reserve(n*4)); CK(ctx->ppB.reserve(n*4)); CK(ctx->ppK.reserve(n*4));
	CK(ctx->ppArcs.reserve(sizeof(int)*4 + (size_t)cap*sizeof(SegArc)));
	int* count = ctx->ppArcs.as<int>();
	SegArc* arcs = (SegArc*)(ctx->ppArcs.as<int>()+4);
	CK(seg_launch_label(depth, width, height, th, ctx->ppA.as<int>(), ctx->ppB.as<int>(), ctx->ppK.as<int>(), arcs, count, cap, s));
	// the condensed graph is resolved on the host: one small read-back (the call synchronises the stream)
	int nArcs = 0;
	CK(cudaMemcpyAsync(&nArcs, count, sizeof(int), cudaMemcpyDeviceToHost, s));
	CK(cudaStreamSynchronize(s));
	if (nArcs > cap) return fail(ctx, B200MVS_ERR_ARG, "remove_small_segments: too many direction-dependent edges in the depth-map");
	int nPatch = 0;
	if (nArcs > 0) {
		std::vector<SegArc> h(nArcs);
		CK(cudaMemcpyAsync(h.data(), arcs, (size_t)nArcs*sizeof(SegArc), cudaMemcpyDeviceToHost, s));
		CK(cudaStreamSynchronize(s));
		// nodes: the components an arc touches; replay of the reference's loop (SceneDensify.cpp:828-895) on them
		struct Node { int label, size, key; std::vector<int> out; int seg = -1; };
		std::vector<Node> nodes;
		std::vector<std::pair<int, int>> index; // (label, node)
		auto node_of = [&](int label, int size, int key) {
			for (auto& p: index) if (p.first == label) return p.second;  // few nodes: linear search is fine ...
			index.push_back({label, (int)nodes.size()});
			Node nd; nd.label = label; nd.size = size; nd.key = key; nodes.push_back(nd);
			return (int)nodes.size()-1;
		};
		if (nArcs > 4096) {  // ... but not for pathological maps: sort once and search
			std::sort(h.begin(), h.end(), [](const SegArc& a, const SegArc& b) { return a.src != b.src ? a.src < b.src : a.dst < b.dst; });
		}
		std::vector<std::pair<int, int>> sortedIndex;
		if (nArcs > 4096) {
			std::vector<std::pair<int, std::pair<int, int>>> all; // label -> (size, key)
			for (auto& a: h) { all.push_back({a.src, {a.srcSize, a.srcKey}}); all.push_back({a.dst, {a.dstSize, a.dstKey}}); }
			std::sort(all.begin(), all.end());
			all.erase(std::unique(all.begin(), all.end(), [](const auto& x, const auto& y) { return x.first == y.first; }), all.end());
			for (auto& e: all) { Node nd; nd.label = e.first; nd.size = e.second.first; nd.key = e.second.second; sortedIndex.push_back({e.first, (int)nodes.size()}); nodes.push_back(nd); }
		}
		auto find_node = [&](int label, int size, int key) {
			if (sortedIndex.empty()) return node_of(label, size, key);
			return std::lower_bound(sortedIndex.begin(), sortedIndex.end(), std::make_pair(label, -1))->second;
		};
		for (auto& a: h) {
			const int u = find_node(a.src, a.srcSize, a.srcKey), v = find_node(a.dst, a.dstSize, a.dstKey);
			nodes[u].out.push_back(v);
		}
		std::vector<int> order(nodes.size());
		for (size_t i = 0; i < order.size(); ++i) order[i] = (int)i;
		std::sort(order.begin(), order.end(), [&](int a, int b) { return nodes[a].key < nodes[b].key; });
		std::vector<int> patch; std::vector<int> stack, members;
		for (int seed: order) {
			if (nodes[seed].seg >= 0) continue;
			// the segment grown from this seed: every unvisited component reachable along one-way edges
			long long total = 0;
			stack.assign(1, seed); members.clear(); nodes[seed].seg = seed;
			while (!stack.empty()) {
				const int u = stack.back(); stack.pop_back();
				members.push_back(u); total += nodes[u].size;
				for (int v: nodes[u].out) if (nodes[v].seg < 0) { nodes[v].seg = seed; stack.push_back(v); }
			}
			for (int u: members) { patch.push_back(nodes[u].label); patch.push_back((int)std::min<long long>(total, 0x7FFFFFFF)); }
		}
		nPatch = (int)patch.size()/2;
		CK(ctx->ppPatch.reserve(patch.size()*sizeof(int)));
		CK(cudaMemcpyAsync(ctx->ppPatch.p, patch.data(), patch.size()*sizeof(int), cudaMemcpyHostToDevice, s));
		CK(cudaStreamSynchronize(s)); // `patch` is a local
	}
	CK(seg_launch_remove(depth, normal, conf, width, height, nSpeckleSize, ctx->ppA.as<int>(), ctx->ppB.as<int>(), ctx->ppPatch.as<int>(), nPatch, s));
	{ int rounds = 1; while ((1<<rounds) < width+height) ++rounds; ctx->launches = 5+2*rounds+(nPatch > 0 ? 1 : 0); }
	return B200MVS_OK;
}

int b200mvs_gap_interpolation_device(b200mvs_ctx* ctx, float* depth, float* normal, float* conf, int width, int height,
	float fDepthDiffThreshold, unsigned nIpolGapSize, void* stream)
{
	if (!ctx) return B200MVS_ERR_ARG;
	if (!depth || width <= 0 || height <= 0 || (size_t)width*height > 0x7FFFFFFFull/3 || !(fDepthDiffThreshold > 0))
		return fail(ctx, B200MVS_ERR_ARG, "gap_interpolation: invalid argument");
	CK(cudaSetDevice(ctx->device));
	const size_t n = (size_t)width*height;
	CK(ctx->ppA.reserve(n*4)); CK(ctx->ppB.reserve(n*4)); CK(ctx->ppN.reserve(n*12));
	const int gap = (int)std::min<unsigned>(nIpolGapSize, (unsigned)std::max(width, height));
	CK(gap_launch(depth, normal, conf, ctx->ppA.as<float>(), ctx->ppN.as<float>(), ctx->ppB.as<float>(), width, height,
		fDepthDiffThreshold*2.5f, gap, stream ? (cudaStream_t)stream : ctx->stream));
	ctx->launches = 2;
	return B200MVS_OK;
}

// host form of the two in-place passes: stage, run, copy back
static int pp_host(b200mvs_ctx* ctx, int which, float* depth, float* normal, float* conf, int width, int height, float th, unsigned arg, b200mvs_stats* stats) {
	if (!ctx) return B200MVS_ERR_ARG;
	if (!depth || width <= 0 || height <= 0) return fail(ctx, B200MVS_ERR_ARG, "post-processing: invalid argument");
	CK(cudaSetDevice(ctx->device));
	cudaStream_t s = ctx->stream;
	const auto t0 = std::chrono::steady_clock::now();
	const size_t n = (size_t)width*height;
	CK(ctx->ppD.reserve(n*4+n*12)); CK(ctx->ppC.reserve(n*4));
	float* dD = ctx->ppD.as<float>(); float* dN = normal ? dD+n : nullptr; float* dC = conf ? ctx->ppC.as<float>() : nullptr;
	CK(cudaMemcpyAsync(dD, depth, n*4, cudaMemcpyHostToDevice, s));
	if (normal) CK(cudaMemcpyAsync(dN, normal, n*12, cudaMemcpyHostToDevice, s));
	if (conf) CK(cudaMemcpyAsync(dC, conf, n*4, cudaMemcpyHostToDevice, s));
	CK(cudaEventRecord(ctx->ev0, s));
	const int rc = which == 0 ? b200mvs_remove_small_segments_device(ctx, dD, dN, dC, width, height, th, arg, s)
		: b200mvs_gap_interpolation_device(ctx, dD, dN, dC, width, height, th, arg, s);
	if (rc) return rc;
	CK(cudaEventRecord(ctx->ev1, s));
	CK(cudaMemcpyAsync(depth, dD, n*4, cudaMemcpyDeviceToHost, s));
	if (normal) CK(cudaMemcpyAsync(normal, dN, n*12, cudaMemcpyDeviceToHost, s));
	if (conf) CK(cudaMemcpyAsync(conf, dC, n*4, cudaMemcpyDeviceToHost, s));
	CK(cudaStreamSynchronize(s));
	if (stats) {
		memset(stats, 0, sizeof(*stats));
		float ms = 0; cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
		const uint64_t b = n*4+(normal ? n*12 : 0)+(conf ? n*4 : 0);
		stats->ms_device = ms; stats->bytes_h2d = b; stats->bytes_d2h = b; stats->kernel_launches = ctx->launches; stats->levels = 1;
		stats->ms_total = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now()-t0).count();
	}
	return B200MVS_OK;
}

int b200mvs_remove_small_segments(b200mvs_ctx* ctx, float* depth, float* normal, float* conf, int width, int height,
	float fDepthDiffThreshold, unsigned nSpeckleSize, b200mvs_stats* stats)
{
	return pp_host(ctx, 0, depth, normal, conf, width, height, fDepthDiffThreshold, nSpeckleSize, stats);
}

int b200mvs_gap_interpolation(b200mvs_ctx* ctx, float* depth, float* normal, float* conf, int width, int height,
	float fDepthDiffThreshold, unsigned nIpolGapSize, b200mvs_stats* stats)
{
	return pp_host(ctx, 1, depth, normal, conf, width, height, fDepthDiffThreshold, nIpolGapSize, stats);
}

// ---- image preparation (SURVEY §8f rank 3): toGray on the device ----
int b200mvs_to_gray_device(b200mvs_ctx* ctx, const uint8_t* image, int width, int height, int stride_bytes, int channels, int bgr,
	float* gray, int gray_stride_bytes, void* stream)
{
	if (!ctx) return B200MVS_ERR_ARG;
	if (!image || !gray || width <= 0 || height <= 0 || (channels != 3 && channels != 4))
		return fail(ctx, B200MVS_ERR_ARG, "to_gray: null pointer, empty image or channel count other than 3 / 4");
	if (stride_bytes == 0) stride_bytes = width*channels;
	if (gray_stride_bytes == 0) gray_stride_bytes = width*4;
	if (stride_bytes < width*channels || gray_stride_bytes < width*4 || (gray_stride_bytes & 3))
		return fail(ctx, B200MVS_ERR_ARG, "to_gray: invalid stride");
	CK(cudaSetDevice(ctx->device));
	CK(rs_launch_to_gray(image, width, height, stride_bytes, channels, bgr != 0, gray, gray_stride_bytes/4, stream ? (cudaStream_t)stream : ctx->stream));
	ctx->launches = 1;
	return B200MVS_OK;
}

// DepthData::ViewData::ScaleImage (libs/MVS/DepthMap.h:193-203): a neighbour whose footprint differs from the reference's by
// 15 % or more is resampled by `scale` — cv::resize(image, Size(), scale, scale, scale > 1 ? INTER_CUBIC : INTER_AREA)
int b200mvs_scaled_size(int width, int height, float scale, int* scaledWidth, int* scaledHeight) {
	if (!scaledWidth || !scaledHeight || width <= 0 || height <= 0 || !(scale > 0)) return B200MVS_ERR_ARG;
	// cv::resize with dsize = Size(): saturate_cast<int>(src.cols * fx) = cvRound
	*scaledWidth = (int)std::nearbyint(width*(double)scale); *scaledHeight = (int)std::nearbyint(height*(double)scale);
	return B200MVS_OK;
}
int b200mvs_scale_image_device(b200mvs_ctx* ctx, const float* image, int width, int height, int stride_bytes, float scale,
	float* scaled, int* applied, void* stream)
{
	if (!ctx) return B200MVS_ERR_ARG;
	if (!image || !scaled || width <= 0 || height <= 0 || !(scale > 0) || (stride_bytes & 3))
		return fail(ctx, B200MVS_ERR_ARG, "scale_image: null pointer, empty image, scale <= 0 or stride not a multiple of 4");
	if (applied) *applied = 0;
	if (std::fabs(scale-1.f) < 0.15f) return B200MVS_OK;  // !NeedScaleImage: the caller keeps the image and its camera
	int dw, dh; b200mvs_scaled_size(width, height, scale, &dw, &dh);
	if (dw <= 0 || dh <= 0) return fail(ctx, B200MVS_ERR_ARG, "scale_image: scaled image is empty");
	CK(cudaSetDevice(ctx->device));
	cudaStream_t s = stream ? (cudaStream_t)stream : ctx->stream;
	const int pitch = stride_bytes ? stride_bytes/4 : width;
	const double inv = 1.0/(double)scale;
	if (scale > 1.f) CK(rs_launch_cubic(image, width, height, pitch, scaled, dw, dh, dw, inv, inv, s));
	else CK(rs_launch_area(image, width, height, pitch, scaled, dw, dh, inv, inv, s));
	ctx->launches = 1;
	if (applied) *applied = 1;
	return B200MVS_OK;
}

} // extern "C"
