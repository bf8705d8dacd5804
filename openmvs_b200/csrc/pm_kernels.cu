// pm_kernels.cu — PatchMatch depth+normal estimation kernels, hand-written for sm_100a.
//
// What they compute (behaviour, not code, follows the reference CPU estimator):
//   pm_score_kernel   pass A  ScoreDepthMapTmp            libs/MVS/SceneDensify.cpp:490-517
//   pm_sweep_kernel   pass B  DepthEstimator::ProcessPixel libs/MVS/DepthMap.cpp:630-852
//                             scored by ScorePixel/ScorePixelImage (DepthMap.cpp:465-626)
//   pm_finalize_kernel pass C EndDepthMapTmp              libs/MVS/SceneDensify.cpp:528-548
//
// Schedule: red-black.  One thread owns one pixel of the active colour; a warp owns 32
// same-colour pixels of one image row (64-pixel span), so the homography-warped taps of
// the 32 lanes fall on 2-3 cache lines of two neighbour-image rows.  The bilateral
// weights of the 5x5 reference patch are computed once per pixel and sweep from a reference
// tile that TMA stages into shared memory, kept in tensor memory (TMEM, one lane per pixel,
// read by tcgen05.ld off the L1 data pipe that the texel gathers bind) and reused by every
// hypothesis x view (80 registers per thread, 24 warps per SM).
// All four 4-neighbours belong to the other colour, so in-place updates are race-free.
// Measured design history and the variants that were dropped: DESIGN.md section 5.1.
#include "pm_common.cuh"
#include <math_constants.h>
#include <cstring>
#include <cuda.h>   // CUtensorMap (type only; the encoder is fetched through cudaGetDriverEntryPoint)

namespace {

constexpr int BLOCK_X = 32;  // lanes: 32 same-colour pixels = 64-pixel span
constexpr int BLOCK_Y = 8;

constexpr int NTHREADS = BLOCK_X*BLOCK_Y;

// Bilateral weights of the 5x5 reference patch (WeightedPatchFix<25>, DepthMap.h:145-155): 50 registers per thread
// less than a register copy.  Two homes with one interface: the scoring code reads tap row i as r[2j] = w, r[2j+1] = tw
// (j = 0..4) through load_row(i, r) and may use r only after wait_row(r).
// PatchW (pass A): shared memory, float2{w,tw}[tap][thread] (conflict-free LDS.64).
struct PatchW {
	float2* s; // &smem[threadIndex]; tap k at s[k*NTHREADS]
	float sumW, normSq0;
	__device__ __forceinline__ void set(int k, float a, float b) { s[k*NTHREADS] = make_float2(a, b); }
	__device__ __forceinline__ void load_row(int i, uint32_t (&r)[10]) const {
		#pragma unroll
		for (int j = 0; j < 5; ++j) {
			const float2 v = s[(5*i+j)*NTHREADS];
			r[2*j] = __float_as_uint(v.x); r[2*j+1] = __float_as_uint(v.y);
		}
	}
	__device__ __forceinline__ void wait_row(uint32_t (&)[10]) const {}
};

// PatchT (the sweep): tensor memory, one TMEM lane per pixel.  A warp reaches only the 32 lanes of its quarter (warp % 4),
// so warps w and w+4 share a quarter at column blocks 0 and 64 of the CTA's 128 columns.  Columns of a block: taps 0..3 of
// row i at 8i..8i+7 ({w, tw} per tap), tap 4 of row i at 40+2i..41+2i.  A tap row is read as one tcgen05.ld .x4 per tap pair
// and one .x2 for the fifth tap, each at its natural alignment (measured 1 % faster per launch than one .x8 + one .x2 per row,
// DESIGN.md §5.1).  tcgen05.ld/st are .sync.aligned: every lane of the warp executes them.
constexpr uint32_t SWEEP_TMEM_COLS = 128;
struct PatchT {
	uint32_t t; // TMEM address: lane quarter << 16 | column block
	float sumW, normSq0;
	__device__ __forceinline__ static uint32_t col(int k) { const int i = k/5, j = k%5; return j < 4 ? 8*i+2*j : 40+2*i; }
	__device__ __forceinline__ void set(int k, float a, float b) {
		asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};"
			:: "r"(t+col(k)), "r"(__float_as_uint(a)), "r"(__float_as_uint(b)) : "memory");
	}
	// volatile: the loads must stay behind the fill's tcgen05.wait::st and must not be hoisted out of the view loop
	__device__ __forceinline__ void load_row(int i, uint32_t (&r)[10]) const {
		asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
			: "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(t+8*i));
		asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
			: "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]) : "r"(t+8*i+4));
		asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(r[8]), "=r"(r[9]) : "r"(t+40+2*i));
	}
	// the registers of an issued tcgen05.ld are undefined until tcgen05.wait::ld: tie them to the wait
	__device__ __forceinline__ void wait_row(uint32_t (&r)[10]) const {
		asm volatile("tcgen05.wait::ld.sync.aligned;"
			: "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]), "+r"(r[9]));
	}
};

// ---- TMA staging of the reference tile ---------------------------------------------------------
// A CTA of the sweep kernel covers 64 x 8 pixels; their 9x9 patches need a (64+8) x (8+8) float tile
// of the reference image.  One elected thread issues a cp.async.bulk.tensor.2d (TMA) into shared
// memory and everybody waits on the mbarrier; out-of-image parts of the box are zero-filled by the
// TMA unit (those pixels are rejected by the patch-inside test anyway).
constexpr int TILE_W = 2*BLOCK_X+2*PM_HALF;   // 72 floats = 288 B (multiple of 16 B)
constexpr int TILE_H = BLOCK_Y+2*PM_HALF;     // 16 rows
constexpr int TILE_BYTES = TILE_W*TILE_H*4;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count) {
	asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
	asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
	asm volatile(
		"{\n"
		".reg .pred p;\n"
		"WAIT_LOOP:\n"
		"mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
		"@p bra WAIT_DONE;\n"
		"bra WAIT_LOOP;\n"
		"WAIT_DONE:\n"
		"}\n" :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
	asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
		:: "r"(smem_u32(dst)), "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar)) : "memory");
}

// FillPixelPatch + GetWeight from the staged tile; (lx, ly) = pixel position inside the tile
template <class PW>
__device__ __forceinline__ void fill_patch_tile(const float* __restrict__ tile, int lx, int ly, PW& p) {
	const float sigmaColor = -1.f/(2.f*0.1f*0.1f);
	const float sigmaSpatial = -1.f/(2.f*9.f);
	const float center = tile[ly*TILE_W + lx];
	float acc = 0.f, sumW = 0.f;
	float w[PM_TEXELS], I[PM_TEXELS];
	#pragma unroll
	for (int i = 0; i < 5; ++i) {
		#pragma unroll
		for (int j = 0; j < 5; ++j) {
			const int dy = 2*i-PM_HALF, dx = 2*j-PM_HALF;
			const float v = tile[(ly+dy)*TILE_W + (lx+dx)];
			const float dI = v-center;
			const float wgt = expf(dI*dI*sigmaColor + float(dx*dx+dy*dy)*sigmaSpatial);
			w[i*5+j] = wgt;
			I[i*5+j] = v;
			acc += v*wgt;
			sumW += wgt;
		}
	}
	const float tm = acc/sumW;
	float nsq = 0.f;
	#pragma unroll
	for (int k = 0; k < PM_TEXELS; ++k) {
		const float t = I[k]-tm;
		const float tw = w[k]*t;
		nsq += tw*t;
		p.set(k, w[k], tw);
	}
	p.sumW = sumW;
	p.normSq0 = nsq;
}

// FillPixelPatch + GetWeight (DepthMap.cpp:422-462, DepthMap.h:403-412) from global memory (pass A, and
// the sweep when no TMA descriptor is available)
template <class PW>
__device__ __forceinline__ void fill_patch(const float* __restrict__ img, int pitch, int x, int y, PW& p) {
	const float sigmaColor = -1.f/(2.f*0.1f*0.1f);
	const float sigmaSpatial = -1.f/(2.f*9.f);
	const float center = __ldg(img + (size_t)y*pitch + x);
	float acc = 0.f, sumW = 0.f;
	float w[PM_TEXELS], I[PM_TEXELS];
	#pragma unroll
	for (int i = 0; i < 5; ++i) {
		#pragma unroll
		for (int j = 0; j < 5; ++j) {
			const int dy = 2*i-PM_HALF, dx = 2*j-PM_HALF;
			const float v = __ldg(img + (size_t)(y+dy)*pitch + (x+dx));
			const float dI = v-center;
			const float wgt = expf(dI*dI*sigmaColor + float(dx*dx+dy*dy)*sigmaSpatial);
			w[i*5+j] = wgt;
			I[i*5+j] = v;
			acc += v*wgt;
			sumW += wgt;
		}
	}
	const float tm = acc/sumW;
	float nsq = 0.f;
	#pragma unroll
	for (int k = 0; k < PM_TEXELS; ++k) {
		const float t = I[k]-tm;
		const float tw = w[k]*t;
		nsq += tw*t;
		p.set(k, w[k], tw);
	}
	p.sumW = sumW;
	p.normSq0 = nsq;
}

struct Hyp {      // one plane hypothesis at the current pixel
	float d;      // depth
	float3 n;     // unit normal, camera space
	float invd;   // 1/d
	float3 ms;    // (n^T Kref^-1) / (n.X0 d)
	float smooth; // product of the smoothness factors (view independent)
};

struct Close {    // the <=4 neighbours used for smoothing (NeighborEstimate, DepthMap.h:300-306)
	float d[4];
	float3 n[4];
	float rx[4], ry[4]; // ray of the neighbour pixel
	unsigned mask;      // bit k set: slot k holds a valid neighbour
};

__device__ __forceinline__ float fast_rcp(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float pow2neg(unsigned i) { return __int_as_float((int)(127u-i)<<23); } // 2^-i, scaleRanges[] (DepthMap.cpp:358-359)
__device__ __forceinline__ float dot3(const float3& a, const float3& b) { return a.x*b.x + a.y*b.y + a.z*b.z; }

// masked bilinear depth sample (TImage::sample with functor, libs/Common/Types.inl:2297-2313)
__device__ __forceinline__ bool sample_depth_masked(const float* __restrict__ img, int pitch, float px, float py, float ref, float& v) {
	const int lx = (int)px, ly = (int)py;
	const float x = px-lx, x1 = 1.f-x, y = py-ly, y1 = 1.f-y;
	const float* r0 = img + (size_t)ly*pitch + lx;
	const float x0y0 = __ldg(r0), x1y0 = __ldg(r0+1), x0y1 = __ldg(r0+pitch), x1y1 = __ldg(r0+pitch+1);
	const bool b00 = fabsf(ref-x0y0)/ref < 0.03f, b10 = fabsf(ref-x1y0)/ref < 0.03f;
	const bool b01 = fabsf(ref-x0y1)/ref < 0.03f, b11 = fabsf(ref-x1y1)/ref < 0.03f;
	if (!b00 && !b10 && !b01 && !b11)
		return false;
	v = y1*(x1*(b00 ? x0y0 : (b10 ? x1y0 : (b01 ? x0y1 : x1y1))) + x*(b10 ? x1y0 : (b00 ? x0y0 : (b11 ? x1y1 : x0y1)))) +
	    y *(x1*(b01 ? x0y1 : (b11 ? x1y1 : (b00 ? x0y0 : x1y0))) + x*(b11 ? x1y1 : (b01 ? x0y1 : (b10 ? x1y0 : x0y0))));
	return true;
}

// The four texels of one warped tap at integer position (lx, ly) of a plain float image (pitch in floats).
// L1 evict-last: the warped footprints of successive hypotheses and of the CTA's other rows overlap, keeping
// them in L1 against the streaming plane/cost traffic is worth 2.5 % (2.73 -> 2.66 ms).
// (measured and dropped, DESIGN.md §5.1: row-pair and float4 quad layouts, column-parity planes, texture gather
//  TLD4, a TLD4/LDG split across views — all slower than plain rows on B200)
__device__ __forceinline__ void fetch_texels(const void* __restrict__ tex, int pitch, int lx, int ly,
	float& v00, float& v10, float& v01, float& v11)
{
	unsigned long long addr;
	const unsigned idx = (unsigned)(ly*pitch + lx);
	asm("mad.wide.u32 %0, %1, %2, %3;" : "=l"(addr) : "r"(idx), "r"(4u), "l"((unsigned long long)tex));
	const float* r0 = (const float*)addr;
	const float* r1 = r0+pitch;
	asm("ld.global.nc.L1::evict_last.f32 %0, [%1];" : "=f"(v00) : "l"(r0));
	asm("ld.global.nc.L1::evict_last.f32 %0, [%1+4];" : "=f"(v10) : "l"(r0));
	asm("ld.global.nc.L1::evict_last.f32 %0, [%1];" : "=f"(v01) : "l"(r1));
	asm("ld.global.nc.L1::evict_last.f32 %0, [%1+4];" : "=f"(v11) : "l"(r1));
}

// ScorePixelImage (DepthMap.cpp:465-564) for one neighbour view.
// The reference rejects a hypothesis as soon as one warped tap leaves the neighbour image
// (1-pixel border).  A homography maps the convex patch quad onto the convex quad of its
// projected corners as long as the depth Z keeps its sign, so "all 25 taps inside" is decided
// once from the 4 corner taps; the tap loop itself is then branch-free and test-free, and the
// loads of a whole tap row are in flight together.  Rejected lanes run the loop on texel (1,1).
// PACK: taps evaluated two at a time with the packed fp32 instructions of sm_100 (FMUL2 / FFMA2 through
// __fmul2_rn / __ffma2_rn): identical roundings (whole-run output bit-identical to the scalar form, photometric
// and geometric passes), about 10 % fewer issue slots per 25 taps.  PACK = false is the debug form.
// have = false: a lane that only keeps its warp converged (TMEM loads are warp-collective); it runs as a rejected lane.
template <bool PACK, bool GEOM, class PW>
__device__ __forceinline__ float score_view(const PMParams& P, const PMView& V, const PW& pt,
	float fx, float fy, float X0x, float X0y, const Hyp& h, float priorF, float priorD, bool have)
{
	// H = A + Hm (n^T Kref^-1)/(n.X0 d); columns 0/1 and the centre point H*(x,y,1)
	float c0x = fmaf(V.Hm[0], h.ms.x, V.A[0]), c0y = fmaf(V.Hm[1], h.ms.x, V.A[3]), c0z = fmaf(V.Hm[2], h.ms.x, V.A[6]);
	float c1x = fmaf(V.Hm[0], h.ms.y, V.A[1]), c1y = fmaf(V.Hm[1], h.ms.y, V.A[4]), c1z = fmaf(V.Hm[2], h.ms.y, V.A[7]);
	const float xc = fmaf(V.Hm[0], h.invd, fmaf(V.A[0], fx, fmaf(V.A[1], fy, V.A[2])));
	const float yc = fmaf(V.Hm[1], h.invd, fmaf(V.A[3], fx, fmaf(V.A[4], fy, V.A[5])));
	const float zc = fmaf(V.Hm[2], h.invd, fmaf(V.A[6], fx, fmaf(V.A[7], fy, V.A[8])));
	// top-left tap, then steps of 2 pixels
	float bx = fmaf(-4.f, c0x+c1x, xc), by = fmaf(-4.f, c0y+c1y, yc), bz = fmaf(-4.f, c0z+c1z, zc);
	c0x *= 2.f; c0y *= 2.f; c0z *= 2.f; c1x *= 2.f; c1y *= 2.f; c1z *= 2.f;
	const float xmax = float(V.w-2), ymax = float(V.h-2);
	bool ok;
	{
		// the four corner taps (0,0) (4,0) (0,4) (4,4)
		const float x1 = fmaf(4.f, c0x, bx), y1 = fmaf(4.f, c0y, by), z1 = fmaf(4.f, c0z, bz);
		const float x2 = fmaf(4.f, c1x, bx), y2 = fmaf(4.f, c1y, by), z2 = fmaf(4.f, c1z, bz);
		const float x3 = fmaf(4.f, c1x, x1), y3 = fmaf(4.f, c1y, y1), z3 = fmaf(4.f, c1z, z1);
		const float zmin = fminf(fminf(bz, z1), fminf(z2, z3)), zmax = fmaxf(fmaxf(bz, z1), fmaxf(z2, z3));
		const float i0 = fast_rcp(bz), i1 = fast_rcp(z1), i2 = fast_rcp(z2), i3 = fast_rcp(z3);
		const float pxmin = fminf(fminf(bx*i0, x1*i1), fminf(x2*i2, x3*i3)), pxmax = fmaxf(fmaxf(bx*i0, x1*i1), fmaxf(x2*i2, x3*i3));
		const float pymin = fminf(fminf(by*i0, y1*i1), fminf(y2*i2, y3*i3)), pymax = fmaxf(fmaxf(by*i0, y1*i1), fmaxf(y2*i2, y3*i3));
		ok = have && (zmin > 0.f || zmax < 0.f) && pxmin >= 1.f && pymin >= 1.f && pxmax <= xmax && pymax <= ymax;
		// NaN anywhere makes a comparison false (fminf/fmaxf drop NaNs, so test them explicitly)
		ok = ok && (bx*i0 == bx*i0) && (x1*i1 == x1*i1) && (x2*i2 == x2*i2) && (x3*i3 == x3*i3)
		        && (by*i0 == by*i0) && (y1*i1 == y1*i1) && (y2*i2 == y2*i2) && (y3*i3 == y3*i3);
	}
	if (!__any_sync(__activemask(), ok))
		return P.thRobust;
	if (!ok) { bx = by = bz = 1.f; c0x = c0y = c0z = c1x = c1y = c1z = 0.f; }
	const void* tex = V.img;
	int pitch = V.pitch;
	// keep the per-view constants in registers (otherwise re-read from the constant bank per tap)
	asm volatile("" : "+r"(pitch), "+l"(tex));
	float sum = 0.f, sumSq = 0.f, num = 0.f;
	const float2 NEG1 = make_float2(-1.f, -1.f);
	#pragma unroll
	for (int i = 0; i < 5; ++i) {
		float X = bx, Y = by, Z = bz;
		uint32_t wr[10]; // weights of tap row i, in flight while the row's texels are fetched
		pt.load_row(i, wr);
		#pragma unroll
		for (int j = 0; j < 5; j += 2) {
			const bool two = j+1 < 5;
			// tap a = j, tap b = j+1 (the fifth tap of a row runs alone in the .x halves)
			const float Xa = X, Ya = Y, Za = Z;
			const float Xb = Xa+c0x, Yb = Ya+c0y, Zb = Za+c0z;
			if (two) { X = Xb+c0x; Y = Yb+c0y; Z = Zb+c0z; }
			const float iza = fast_rcp(Za), izb = two ? fast_rcp(Zb) : 0.f;
			float2 PX, PY;
			if (PACK && two) { PX = __fmul2_rn(make_float2(Xa, Xb), make_float2(iza, izb)); PY = __fmul2_rn(make_float2(Ya, Yb), make_float2(iza, izb)); }
			else { PX = make_float2(Xa*iza, Xb*izb); PY = make_float2(Ya*iza, Yb*izb); }
			const int lxa = __float2int_rz(PX.x), lya = __float2int_rz(PY.x);
			const int lxb = two ? __float2int_rz(PX.y) : 1, lyb = two ? __float2int_rz(PY.y) : 1;
			const float2 FLX = make_float2((float)lxa, (float)lxb), FLY = make_float2((float)lya, (float)lyb);
			float2 AX, AY;
			if (PACK && two) { AX = __ffma2_rn(FLX, NEG1, PX); AY = __ffma2_rn(FLY, NEG1, PY); }
			else { AX = make_float2(PX.x-FLX.x, PX.y-FLX.y); AY = make_float2(PY.x-FLY.x, PY.y-FLY.y); }
			float2 V00, V10, V01, V11;
			fetch_texels(tex, pitch, lxa, lya, V00.x, V10.x, V01.x, V11.x);
			if (two) fetch_texels(tex, pitch, lxb, lyb, V00.y, V10.y, V01.y, V11.y);
			else { V00.y = V10.y = V01.y = V11.y = 0.f; }
			float2 DT, TOP, DB, BOT, DV, VV;
			if (PACK && two) {
				DT = __ffma2_rn(V00, NEG1, V10); TOP = __ffma2_rn(AX, DT, V00);
				DB = __ffma2_rn(V01, NEG1, V11); BOT = __ffma2_rn(AX, DB, V01);
				DV = __ffma2_rn(TOP, NEG1, BOT); VV = __ffma2_rn(AY, DV, TOP);
			} else {
				TOP = make_float2(fmaf(AX.x, V10.x-V00.x, V00.x), fmaf(AX.y, V10.y-V00.y, V00.y));
				BOT = make_float2(fmaf(AX.x, V11.x-V01.x, V01.x), fmaf(AX.y, V11.y-V01.y, V01.y));
				VV = make_float2(fmaf(AY.x, BOT.x-TOP.x, TOP.x), fmaf(AY.y, BOT.y-TOP.y, TOP.y));
			}
			if (j == 0)
				pt.wait_row(wr);
			{
				const float2 wk = make_float2(__uint_as_float(wr[2*j]), __uint_as_float(wr[2*j+1]));
				const float vw = VV.x*wk.x;
				sum += vw; sumSq = fmaf(VV.x, vw, sumSq); num = fmaf(VV.x, wk.y, num);
			}
			if (two) {
				const float2 wk = make_float2(__uint_as_float(wr[2*j+2]), __uint_as_float(wr[2*j+3]));
				const float vw = VV.y*wk.x;
				sum += vw; sumSq = fmaf(VV.y, vw, sumSq); num = fmaf(VV.y, wk.y, num);
			}
		}
		bx += c1x; by += c1y; bz += c1z;
	}
	const bool bad = !ok;
	if (bad)
		return P.thRobust;
	const float normSq1 = sumSq - sum*sum/pt.sumW;
	const float nrmSq = pt.normSq0*normSq1;
	if (nrmSq <= 1e-16f)
		return P.thRobust;
	const float ncc = fminf(fmaxf(num/sqrtf(nrmSq), -1.f), 1.f);
	float score = (1.f-ncc)*h.smooth;
	if (GEOM) {
		if (V.dmap) {
			// forward/backward reprojection through the neighbour's depth-map (DepthMap.cpp:535-551)
			float consistency = 4.f;
			const float Xx = X0x*h.d, Xy = X0y*h.d, Xz = h.d;
			const float X1x = V.Tl[0]*Xx + V.Tl[1]*Xy + V.Tl[2]*Xz + V.Tm[0];
			const float X1y = V.Tl[3]*Xx + V.Tl[4]*Xy + V.Tl[5]*Xz + V.Tm[1];
			const float X1z = V.Tl[6]*Xx + V.Tl[7]*Xy + V.Tl[8]*Xz + V.Tm[2];
			if (X1z > 0.f) {
				const float x1x = X1x/X1z, x1y = X1y/X1z;
				if (x1x >= 1.f && x1y >= 1.f && x1x <= float(V.dw-2) && x1y <= float(V.dh-2)) {
					float depth1;
					if (sample_depth_masked(V.dmap, V.dpitch, x1x, x1y, X1z, depth1)) {
						const float Px = x1x*depth1, Py = x1y*depth1, Pz = depth1;
						const float Bx = V.Tr[0]*Px + V.Tr[1]*Py + V.Tr[2]*Pz + V.Tn[0];
						const float By = V.Tr[3]*Px + V.Tr[4]*Py + V.Tr[5]*Pz + V.Tn[1];
						const float Bz = V.Tr[6]*Px + V.Tr[7]*Py + V.Tr[8]*Pz + V.Tn[2];
						const float ex = fx-Bx/Bz, ey = fy-By/Bz;
						const float dist = sqrtf(ex*ex + ey*ey);
						consistency = fminf(sqrtf(dist*(dist+2.f)), consistency);
					}
				}
			}
			score += P.geomWeight*consistency;
		}
	}
	if (priorD > 0.f) {
		// low-resolution depth prior (DepthMap.cpp:552-561)
		const float deltaDepth = fminf(fabsf(priorD-h.d)/priorD, 0.5f);
		score = (1.f-priorF)*score + priorF*deltaDepth;
	}
	return fminf(2.f, score);
}

// ScorePixel (DepthMap.cpp:567-626): MINMEAN over the views; also reports the two best views
template <bool PACK, bool GEOM, class PW>
__device__ __forceinline__ float score_pixel(const PMParams& P, const PW& pt,
	float fx, float fy, float X0x, float X0y, const Hyp& h, float priorF, float priorD, bool have, uint32_t& best)
{
	float s0 = CUDART_INF_F, s1 = CUDART_INF_F;
	int i0 = 255, i1 = 255;
	#pragma unroll 1
	for (int v = 0; v < P.nViews; ++v) {
		const float s = score_view<PACK, GEOM>(P, P.views[v], pt, fx, fy, X0x, X0y, h, priorF, priorD, have);
		if (s < s0) { s1 = s0; i1 = i0; s0 = s; i0 = v; }
		else if (s < s1) { s1 = s; i1 = v; }
	}
	if (P.nViews <= 1 || s1 >= P.thRobust) {
		best = 0xFFFFFF00u | (uint32_t)i0;
		return s0;
	}
	best = 0xFFFF0000u | ((uint32_t)i1<<8) | (uint32_t)i0;
	return (s0+s1)*0.5f;
}

// build a hypothesis: homography terms + smoothness factor over the close neighbours
// (InitPlane DepthMap.cpp:963-971 and the smoothness loop DepthMap.cpp:522-534)
__device__ __forceinline__ void make_hyp(const PMParams& P, float X0x, float X0y, float d, const float3& n,
	const Close& cl, bool useClose, Hyp& h)
{
	h.d = d; h.n = n;
	h.invd = 1.f/d;
	const float nX0 = n.x*X0x + n.y*X0y + n.z;
	const float s = 1.f/(nX0*d);
	h.ms = make_float3(n.x*P.ifx*s, (n.x*P.sk + n.y*P.ify)*s, (n.x*P.ox + n.y*P.oy + n.z)*s);
	float smooth = 1.f;
	if (useClose) {
		const float planeD = -d*nX0;
		const float nn = dot3(n, n);
		#pragma unroll
		for (int k = 0; k < 4; ++k) {
			if (cl.mask & (1u<<k)) {
				const float dist = (n.x*cl.rx[k] + n.y*cl.ry[k] + n.z)*cl.d[k] + planeD;
				const float rd = dist/d;
				const float factorDepth = expf(rd*rd*P.smoothSigmaDepth);
				float ca = dot3(n, cl.n[k])/sqrtf(nn*dot3(cl.n[k], cl.n[k]));
				ca = fminf(fmaxf(ca, -1.f), 1.f);
				const float ang = acosf(ca);
				const float factorNormal = expf(ang*ang*P.smoothSigmaNormal);
				smooth *= (1.f-P.smoothBonusDepth*factorDepth)*(1.f-P.smoothBonusNormal*factorNormal);
			}
		}
	}
	h.smooth = smooth;
}

__device__ __forceinline__ float3 dir2normal(float a, float b) {
	float sa, ca, sb, cb;
	sincosf(a, &sa, &ca);
	sincosf(b, &sb, &cb);
	return make_float3(ca*sb, sa*sb, cb);
}
// RandomNormal (DepthMap.h:439-444)
__device__ __forceinline__ float3 random_normal(float u1, float u2, float X0x, float X0y) {
	const float kPI = 3.14159265358979323846f;
	const float a = 0.f + (kPI-0.f)*u1;
	const float b = 0.5f*kPI + (kPI-0.5f*kPI)*u2;
	float3 n = dir2normal(a, b);
	if (n.x*X0x + n.y*X0y + n.z > 0.f)
		n = make_float3(-n.x, -n.y, -n.z);
	return n;
}
// CorrectNormal (DepthMap.h:447-453): rotate n to at most ~90 deg from the viewing ray
__device__ __forceinline__ void correct_normal(float3& n, float X0x, float X0y) {
	const float cosAngLen = n.x*X0x + n.y*X0y + n.z;
	if (cosAngLen >= 0.f) {
		const float kPI = 3.14159265358979323846f;
		const float vlen = sqrtf(X0x*X0x + X0y*X0y + 1.f);
		const float ang = fminf((acosf(cosAngLen/vlen) - 0.5f*kPI)*1.01f, -0.001f);
		float3 w = make_float3(n.y*1.f - n.z*X0y, n.z*X0x - n.x*1.f, n.x*X0y - n.y*X0x); // n x viewDir
		const float inv = 1.f/sqrtf(dot3(w, w));
		w.x *= inv; w.y *= inv; w.z *= inv;
		float s, c;
		sincosf(ang, &s, &c);
		// Rodrigues: R v = v + s (w x v) + (1-c) w x (w x v)
		const float3 wv = make_float3(w.y*n.z - w.z*n.y, w.z*n.x - w.x*n.z, w.x*n.y - w.y*n.x);
		const float3 wwv = make_float3(w.y*wv.z - w.z*wv.y, w.z*wv.x - w.x*wv.z, w.x*wv.y - w.y*wv.x);
		const float c1 = 1.f-c;
		n = make_float3(n.x + s*wv.x + c1*wwv.x, n.y + s*wv.y + c1*wwv.y, n.z + s*wv.z + c1*wwv.z);
	}
}

// The cost field doubles as the "changed" memory of the red-black schedule: the sign bit of a pixel's stored
// cost is set when its last update left its plane unchanged (costs are >= 0, so the bit is free; -0.f counts).
__device__ __forceinline__ bool cost_unchanged(float c) { return (__float_as_uint(c)>>31) != 0u; }

// ------------------------------------------------------------------------------------
// pass A: score the initial estimate of every pixel (random where invalid)
template <bool PACK, bool GEOM>
__global__ void __launch_bounds__(BLOCK_X*BLOCK_Y, 3)
pm_score_kernel(const __grid_constant__ PMParams P)
{
	extern __shared__ float2 smemW[];
	const int x = blockIdx.x*BLOCK_X + threadIdx.x;
	const int y = blockIdx.y*BLOCK_Y + threadIdx.y;
	if (x >= P.W || y >= P.H)
		return;
	const size_t idx = (size_t)y*P.W + x;
	const bool inside = x >= PM_HALF && y >= PM_HALF && x < P.W-PM_HALF && y < P.H-PM_HALF;
	PatchW pt;
	pt.s = smemW + threadIdx.y*BLOCK_X + threadIdx.x;
	float priorD = 0.f, priorF = 0.f;
	// ignore-mask (DepthData::ApplyIgnoreMask, DepthMap.cpp:215-230; masked pixels are not in the pixel list,
	// DepthMap.cpp:343): depth / normal zero, never scored.  Internally their cost is 2 like every rejected pixel.
	bool ok = inside && !(P.mask && P.mask[(size_t)y*P.maskPitch + x] == 0);
	if (ok) {
		fill_patch(P.img0, P.pitch0, x, y, pt);
		if (P.lowres)
			priorD = fmaxf(__ldg(P.lowres + idx), 0.f);
		if (pt.normSq0 < P.thMagnitudeSq && !(priorD > 0.f))
			ok = false;
	}
	if (!ok) {
		P.plane[idx] = make_float4(0.f, 0.f, 0.f, 0.f);
		P.cost[idx] = 2.f;
		if (P.bestViews) P.bestViews[idx] = 0xFFFFFFFFu;
		return;
	}
	if (priorD > 0.f)
		priorF = expf(pt.normSq0*(-1.f/0.02f));
	const float fx = float(x), fy = float(y);
	const float X0x = fx*P.ifx + fy*P.sk + P.ox, X0y = fy*P.ify + P.oy;
	float4 pl = P.plane[idx];
	float3 n = make_float3(pl.x, pl.y, pl.z);
	float d = pl.w;
	const uint4 r = philox4x32_10(make_uint4((uint32_t)idx, 0u, 0u, 0u), make_uint2(P.seed, 0xB200C0DEu));
	if (!(P.dMin <= d && d < P.dMax)) {
		const float s = P.dMinSqr + (P.dMaxSqr-P.dMinSqr)*u32_to_unit(r.x);
		d = s*s;
		n = random_normal(u32_to_unit(r.y), u32_to_unit(r.z), X0x, X0y);
	} else if (n.x*X0x + n.y*X0y + n.z >= 0.f) {
		n = random_normal(u32_to_unit(r.x), u32_to_unit(r.y), X0x, X0y);
	}
	Close cl; cl.mask = 0;
	Hyp h;
	make_hyp(P, X0x, X0y, d, n, cl, false, h);
	uint32_t best;
	const float c = score_pixel<PACK, GEOM>(P, pt, fx, fy, X0x, X0y, h, priorF, priorD, true, best);
	P.plane[idx] = make_float4(n.x, n.y, n.z, d);
	P.cost[idx] = c;
	if (P.bestViews) P.bestViews[idx] = best;
}

// ------------------------------------------------------------------------------------
// pass B: one red-black half-sweep (ProcessPixel, DepthMap.cpp:630-852, on the engine schedule):
//   1. gather the four 4-neighbours (smoothing set "close", DepthMap.cpp:641-766) and, per direction, the
//      propagation candidate: the pixel of the other colour at distance 1, 3, .. 2*farRings+1 with the lowest
//      stored cost (the nearest on ties) — the red-black stand-in for the transport along the scanline that
//      the reference's sequential sweep performs within one iteration;
//   2. test the candidates' planes (InterpolatePixel + CorrectNormal), skipping a direction whose candidates
//      all kept their plane in their last update (they lost against this pixel one sweep ago) — P.skipUnchanged;
//   3. the refinement state machine (DepthMap.cpp:800-852).
// Every lane keeps its own to-do list of directions, so a warp runs max-over-lanes(list length) test steps.
//
// The TMEM loads of the scoring code are warp-collective, so every lane of a warp that has a pixel to update runs the whole
// loop: a lane whose pixel is on the border, masked out or textureless is not `live` (it never has a hypothesis and stores
// nothing), and a lane without a hypothesis in a step scores its current plane as a rejected lane and drops the result.
template <bool PACK, bool GEOM>
__device__ __forceinline__ void sweep_pixel(const PMParams& P, const float* __restrict__ tile, uint32_t tmem, int x, int y, bool live)
{
	const int W = P.W, H = P.H;
	const size_t idx = (size_t)y*W + x;
	PatchT pt;
	pt.t = tmem;
	// a dead lane fills from any in-image patch (the warp has a live pixel, so the image is at least 9 x 9)
	if (P.tma)
		fill_patch_tile(tile, 2*(int)threadIdx.x + ((y+P.colour)&1) + PM_HALF, (int)threadIdx.y + PM_HALF, pt);
	else
		fill_patch(P.img0, P.pitch0, live ? x : PM_HALF, live ? y : PM_HALF, pt);
	asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
	float priorD = 0.f, priorF = 0.f;
	if (live && P.lowres)
		priorD = fmaxf(__ldg(P.lowres + idx), 0.f);
	if (pt.normSq0 < P.thMagnitudeSq && !(priorD > 0.f))
		live = false;
	if (priorD > 0.f)
		priorF = expf(pt.normSq0*(-1.f/0.02f));
	const float fx = float(x), fy = float(y);
	const float X0x = fx*P.ifx + fy*P.sk + P.ox, X0y = fy*P.ify + P.oy;

	// neighbours: causal pair of the sweep direction first (DepthMap.cpp:641-766)
	const int dir = P.sweep & 1;
	const int nProp = P.propagation, farRings = P.farRings;
	Close cl; cl.mask = 0;
	unsigned todo = 0;    // bit k: direction k has a candidate to test
	unsigned farSel = 0;  // 2 bits per direction: ring of the candidate (distance 2*ring+1)
	#pragma unroll
	for (int k = 0; k < 4; ++k) {
		// dir 0: left, up, right, down;  dir 1: right, down, left, up
		const int kk = dir ? (k^2) : k;
		const int ox = (kk == 0) ? -1 : (kk == 2) ? 1 : 0;
		const int oy = (kk == 1) ? -1 : (kk == 3) ? 1 : 0;
		const bool ok = live && ((kk == 0) ? (x > PM_HALF) : (kk == 1) ? (y > PM_HALF) : (kk == 2) ? (x < W-PM_HALF) : (y < H-PM_HALF));
		cl.d[k] = 0.f; cl.n[k] = make_float3(0.f, 0.f, 0.f); cl.rx[k] = 0.f; cl.ry[k] = 0.f;
		if (ok) {
			const size_t nidx = (size_t)(y+oy)*W + (x+ox);
			const float4 np = P.plane[nidx];
			const float nc = P.cost[nidx];
			bool changed = !cost_unchanged(nc);
			float bestC = 3.f;
			if (np.w > 0.f) {
				cl.mask |= 1u<<k;
				cl.d[k] = np.w; cl.n[k] = make_float3(np.x, np.y, np.z);
				const float nfx = float(x+ox), nfy = float(y+oy);
				cl.rx[k] = nfx*P.ifx + nfy*P.sk + P.ox; cl.ry[k] = nfy*P.ify + P.oy;
				bestC = fabsf(nc);
			}
			if (k < nProp) {
				unsigned ring = 0;
				for (int f = 1; f <= farRings; ++f) {
					const int qx = x+ox*(2*f+1), qy = y+oy*(2*f+1);
					if (qx < PM_HALF || qy < PM_HALF || qx >= W-PM_HALF || qy >= H-PM_HALF)
						break;
					const float fc = P.cost[(size_t)qy*W + qx];
					changed = changed || !cost_unchanged(fc);
					if (fabsf(fc) < bestC) { bestC = fabsf(fc); ring = (unsigned)f; }
				}
				if (bestC < P.keep && (changed || !P.skipUnchanged)) {
					todo |= 1u<<k;
					farSel |= ring<<(2*k);
				}
			}
		}
	}
	const float4 pl = live ? P.plane[idx] : make_float4(0.f, 0.f, -1.f, 1.f); // a dead lane: a finite plane to score
	float conf = live ? fabsf(P.cost[idx]) : 0.f;
	float depth = pl.w;
	float3 normal = make_float3(pl.x, pl.y, pl.z);
	uint32_t bestViews = (live && P.bestViews) ? P.bestViews[idx] : 0xFFFFFFFFu;

	// ---- propagation (DepthMap.cpp:775-799), then the refinement state machine (DepthMap.cpp:800-852) ----
	// One loop and one copy of the scoring code for both: a lane first pops its propagation candidates, then runs its
	// refinement tries; lanes with fewer candidates start refining while the others still propagate.  Per pixel the order is
	// the reference's (candidates, then tries), and every try has its own Philox slot (restart try k: slot k, refinement try
	// k: slot nR+k), so the result does not depend on the step at which a lane executes it.
	// evalCap > 0 (engine schedule, b200mvs_params.nEvalCap): a pixel that tests c candidates spends at most
	// max(1, evalCap - c) tries of each kind — pixels whose four directions all changed give up their finest perturbation.
	const int nR = P.nRandomIters;
	const int nRl = P.evalCap > 0 ? min(nR, max(P.evalCap-__popc(todo), 1)) : nR;
	const uint2 key = make_uint2(P.seed, 0xB200C0DEu);
	const uint32_t phase = 1u + (uint32_t)P.sweep;
	int mode = live ? 0 : 3;    // 0 undecided, 1 restart (fully random), 2 refine, 3 done
	bool entered = !live;       // the state machine has taken its first decision
	bool useClose = true;
	unsigned idxScale = 0;
	float scaleRange = 1.f, depthRange = 0.f, pa = 0.f, pb = 0.f;
	int nRestart = 0, nRefine = 0; // tries spent
	#pragma unroll 1
	for (;;) {
		bool have = false, isRefine = false, alive = false, uc = true;
		float hd = 0.f, na = 0.f, nb = 0.f; float3 hn = make_float3(0.f, 0.f, 1.f);
		if (todo != 0u) {
			const int k = __ffs((int)todo)-1;
			todo &= todo-1u;
			const int kk = dir ? (k^2) : k;
			const int dist = 2*(int)((farSel>>(2*k))&3u)+1;
			const int qx = x + ((kk == 0) ? -dist : (kk == 2) ? dist : 0);
			const int qy = y + ((kk == 1) ? -dist : (kk == 3) ? dist : 0);
			const float4 qp = P.plane[(size_t)qy*W + qx];
			// InterpolatePixel (DepthMap.cpp:915-959): the candidate's plane intersected with this pixel's ray,
			// restricted to the row / column; the reference's ray coordinates carry no skew term
			const bool vertical = (kk & 1) != 0;
			const float ncomp = vertical ? qp.y : qp.x;
			const float nx1 = vertical ? X0y : fmaf(fx, P.ifx, P.ox0);
			const float x1 = vertical ? fmaf(float(qy), P.ify, P.oy) : fmaf(float(qx), P.ifx, P.ox0);
			const float denom = qp.z + nx1*ncomp;
			hd = qp.w;
			if (!(fabsf(denom) < 0.0001f)) {
				const float dn = qp.w*(qp.z + x1*ncomp)/denom;
				if (P.dMin <= dn && dn < P.dMax)
					hd = dn;
			}
			hn = make_float3(qp.x, qp.y, qp.z);
			correct_normal(hn, X0x, X0y);
			have = true; alive = true;
		} else {
			if (!entered || (mode == 1 && conf < P.thConfRand)) {
				// RefineIters: choose the perturbation scale from the current score
				entered = true;
				bool toRefine = true;
				if (conf <= P.thConfSmall) idxScale = 2;
				else if (conf <= P.thConfBig) idxScale = 1;
				else if (conf >= P.thConfRand && mode == 0) { mode = 1; useClose = false; toRefine = false; }
				if (toRefine) {
					mode = 2;
					scaleRange = pow2neg(idxScale);
					depthRange = depth*P.depthRatio;
					pa = atan2f(normal.y, normal.x);
					pb = acosf(normal.z);
				}
			}
			if (mode == 1 && nRestart >= nRl) mode = 3; // all random tries failed: no refinement this sweep
			alive = (mode == 1) || (mode == 2 && nRefine < nRl);
			uc = useClose;
			if (mode == 1) {
				// completely random plane (DepthMap.cpp:810-825)
				const uint4 r = philox4x32_10(make_uint4((uint32_t)idx, phase, (uint32_t)nRestart, 0u), key);
				++nRestart;
				const float s = P.dMinSqr + (P.dMaxSqr-P.dMinSqr)*u32_to_unit(r.x);
				hd = s*s;
				hn = random_normal(u32_to_unit(r.y), u32_to_unit(r.z), X0x, X0y);
				have = true;
			} else if (mode == 2 && nRefine < nRl) {
				// perturb around the current estimate (DepthMap.cpp:832-851)
				const uint4 r = philox4x32_10(make_uint4((uint32_t)idx, phase, (uint32_t)(nR+nRefine), 0u), key);
				++nRefine;
				hd = depth + depthRange*scaleRange*(2.f*u32_to_unit(r.x)-1.f);
				if (P.dMin <= hd && hd < P.dMax) {
					na = pa + P.angle1Range*scaleRange*(2.f*u32_to_unit(r.y)-1.f);
					nb = pb + P.angle2Range*scaleRange*(2.f*u32_to_unit(r.z)-1.f);
					hn = dir2normal(na, nb);
					have = hn.x*X0x + hn.y*X0y + hn.z < 0.f;
					isRefine = true;
				}
			}
		}
		if (!__any_sync(__activemask(), alive))
			break;
		if (!__any_sync(__activemask(), have))
			continue;
		if (!have) { hd = depth; hn = normal; }
		Hyp h;
		make_hyp(P, X0x, X0y, hd, hn, cl, uc, h);
		uint32_t bv;
		const float nconf = score_pixel<PACK, GEOM>(P, pt, fx, fy, X0x, X0y, h, priorF, priorD, have, bv);
		if (have && conf > nconf) {
			conf = nconf; depth = hd; normal = hn; bestViews = bv;
			if (isRefine) {
				pa = na; pb = nb;
				++idxScale;
				scaleRange = pow2neg(idxScale);
			}
		}
	}
	if (!live)
		return;
	const bool same = depth == pl.w && normal.x == pl.x && normal.y == pl.y && normal.z == pl.z;
	P.plane[idx] = make_float4(normal.x, normal.y, normal.z, depth);
	P.cost[idx] = (same && P.skipUnchanged) ? -conf : conf;
	if (P.bestViews) P.bestViews[idx] = bestViews;
}

// MINB: resident CTAs per SM the register allocation aims at: 3 (80 registers, the default) or 4 (64 registers: one more CTA of
// latency hiding against more spill traffic — b200mvs_debug.sweepFourCtas, measured in profiles/pm_4ctas_r02.txt: slower).
// TMEM: SWEEP_TMEM_COLS columns per CTA, so 3 or 4 resident CTAs fit the 512 columns of an SM whichever launches they belong to.
template <bool PACK, bool GEOM, int MINB>
__global__ void __launch_bounds__(BLOCK_X*BLOCK_Y, MINB)
pm_sweep_kernel(const __grid_constant__ PMParams P, const __grid_constant__ CUtensorMap tmapRef)
{
	extern __shared__ __align__(128) unsigned char smemRaw[];
	// [ reference tile | mbarrier | TMEM address ]
	float* tile = (float*)smemRaw;
	uint64_t* bar = (uint64_t*)(tile + TILE_W*TILE_H);
	uint32_t* sTmem = (uint32_t*)(bar+1);
	const int tid = threadIdx.y*BLOCK_X + threadIdx.x, warp = tid>>5;
	if (warp == 0) {
		asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(sTmem)), "r"(SWEEP_TMEM_COLS) : "memory");
		asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
	}
	if (P.tma && tid == 32) {
		mbar_init(bar, 1);
		asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); // make the init visible to the async proxy
	}
	asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
	__syncthreads();
	asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
	const uint32_t tmem = *sTmem + ((uint32_t)(32*(warp&3))<<16) + (warp >= 4 ? 64u : 0u);
	if (P.tma) {
		if (tid == 0) {
			mbar_expect_tx(bar, TILE_BYTES);
			tma_load_2d(tile, &tmapRef, (int)blockIdx.x*(2*BLOCK_X)-PM_HALF, (int)blockIdx.y*BLOCK_Y-PM_HALF, bar);
		}
		mbar_wait(bar, 0);
	}
	const int y = blockIdx.y*BLOCK_Y + threadIdx.y;
	const int x = blockIdx.x*(2*BLOCK_X) + 2*threadIdx.x + ((y+P.colour)&1);
	const bool live = x >= PM_HALF && y >= PM_HALF && x < P.W-PM_HALF && y < P.H-PM_HALF &&
		!(P.mask && P.mask[(size_t)y*P.maskPitch + x] == 0);
	if (__any_sync(0xFFFFFFFFu, live))   // warp-uniform: a warp without a pixel to update has nothing to do
		sweep_pixel<PACK, GEOM>(P, tile, tmem, x, y, live);
	asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
	__syncthreads();
	if (warp == 0)
		asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(*sTmem), "r"(SWEEP_TMEM_COLS) : "memory");
}

// pass C: threshold and convert cost to confidence (EndDepthMapTmp).  viewsMap: the (at most two) views of the
// MINMEAN score in ascending order, 255 padding — the order PatchMatchCUDA.cpp:374-391 emits its view ids in
__global__ void pm_finalize_kernel(int n, float keep, const float4* __restrict__ plane, const float* __restrict__ cost,
	const uint32_t* __restrict__ bestViews, float* __restrict__ depth, float* __restrict__ normal, float* __restrict__ conf,
	uint32_t* __restrict__ viewsMap)
{
	const int i = blockIdx.x*blockDim.x + threadIdx.x;
	if (i >= n) return;
	const float4 p = plane[i];
	const float c = fabsf(cost[i]);
	float d = p.w, cf; float3 nn = make_float3(p.x, p.y, p.z);
	uint32_t bv = bestViews ? bestViews[i] : 0xFFFFFFFFu;
	if (d <= 0.f || c >= keep) {
		d = 0.f; cf = 0.f; nn = make_float3(0.f, 0.f, 0.f); bv = 0xFFFFFFFFu;
	} else {
		cf = c >= 1.f ? 0.f : 1.f-c;
		const uint32_t a = bv & 0xFFu, b = (bv>>8) & 0xFFu;
		bv = 0xFFFF0000u | (max(a, b)<<8) | min(a, b);
	}
	depth[i] = d; conf[i] = cf;
	normal[3*(size_t)i] = nn.x; normal[3*(size_t)i+1] = nn.y; normal[3*(size_t)i+2] = nn.z;
	if (viewsMap) viewsMap[i] = bv;
}

__global__ void pm_pack_kernel(int n, const float* __restrict__ depth, const float* __restrict__ normal, float4* __restrict__ plane) {
	const int i = blockIdx.x*blockDim.x + threadIdx.x;
	if (i >= n) return;
	plane[i] = make_float4(normal[3*(size_t)i], normal[3*(size_t)i+1], normal[3*(size_t)i+2], depth[i]);
}
__global__ void pm_unpack_kernel(int n, const float4* __restrict__ plane, float* __restrict__ depth, float* __restrict__ normal) {
	const int i = blockIdx.x*blockDim.x + threadIdx.x;
	if (i >= n) return;
	const float4 p = plane[i];
	depth[i] = p.w;
	normal[3*(size_t)i] = p.x; normal[3*(size_t)i+1] = p.y; normal[3*(size_t)i+2] = p.z;
}

// ---- host launchers ---------------------------------------------------------------------
constexpr size_t W_BYTES = (size_t)PM_TEXELS*NTHREADS*sizeof(float2);
constexpr size_t SWEEP_SMEM = TILE_BYTES + 16;   // tile, mbarrier, TMEM address: below the 48 KB default, no opt-in

template <bool PACK, bool GEOM>
cudaError_t configure_one() {
	return cudaFuncSetAttribute(pm_score_kernel<PACK, GEOM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)W_BYTES);
}

} // namespace

// Opt the kernels of the current device into their dynamic shared memory sizes.  Called by b200mvs_create for its
// device (function attributes are per device; the call is idempotent and safe from several host threads).
cudaError_t pm_configure_device() {
	cudaError_t e;
	if ((e = configure_one<true, false>()) != cudaSuccess) return e;
	if ((e = configure_one<true, true>()) != cudaSuccess) return e;
	if ((e = configure_one<false, false>()) != cudaSuccess) return e;
	return configure_one<false, true>();
}
cudaError_t pm_launch_score(const PMParams& P, bool pack, bool geom, cudaStream_t s) {
	dim3 block(BLOCK_X, BLOCK_Y), grid((P.W+BLOCK_X-1)/BLOCK_X, (P.H+BLOCK_Y-1)/BLOCK_Y);
	if (pack) { if (geom) pm_score_kernel<true, true><<<grid, block, W_BYTES, s>>>(P); else pm_score_kernel<true, false><<<grid, block, W_BYTES, s>>>(P); }
	else { if (geom) pm_score_kernel<false, true><<<grid, block, W_BYTES, s>>>(P); else pm_score_kernel<false, false><<<grid, block, W_BYTES, s>>>(P); }
	return cudaGetLastError();
}
// tmapRef: TMA descriptor of the reference image with box {72, 16} (pm_tma_box), or null (P.tma must be 0)
template <int MINB>
static void launch_sweep(const PMParams& P, const CUtensorMap& map, bool pack, bool geom, dim3 grid, dim3 block, cudaStream_t s) {
	if (pack) { if (geom) pm_sweep_kernel<true, true, MINB><<<grid, block, SWEEP_SMEM, s>>>(P, map); else pm_sweep_kernel<true, false, MINB><<<grid, block, SWEEP_SMEM, s>>>(P, map); }
	else { if (geom) pm_sweep_kernel<false, true, MINB><<<grid, block, SWEEP_SMEM, s>>>(P, map); else pm_sweep_kernel<false, false, MINB><<<grid, block, SWEEP_SMEM, s>>>(P, map); }
}
cudaError_t pm_launch_sweep(const PMParams& P, const void* tmapRef, bool pack, bool geom, bool fourCtas, cudaStream_t s) {
	dim3 block(BLOCK_X, BLOCK_Y), grid((P.W+2*BLOCK_X-1)/(2*BLOCK_X), (P.H+BLOCK_Y-1)/BLOCK_Y);
	CUtensorMap map; memset(&map, 0, sizeof(map));
	if (tmapRef) memcpy(&map, tmapRef, sizeof(map));
	if (fourCtas) launch_sweep<4>(P, map, pack, geom, grid, block, s);
	else launch_sweep<3>(P, map, pack, geom, grid, block, s);
	return cudaGetLastError();
}
void pm_tma_box(int* w, int* h) { *w = TILE_W; *h = TILE_H; }
cudaError_t pm_launch_finalize(int n, float keep, const float4* plane, const float* cost, const uint32_t* bestViews,
	float* depth, float* normal, float* conf, uint32_t* viewsMap, cudaStream_t s) {
	pm_finalize_kernel<<<(n+255)/256, 256, 0, s>>>(n, keep, plane, cost, bestViews, depth, normal, conf, viewsMap);
	return cudaGetLastError();
}
cudaError_t pm_launch_pack(int n, const float* depth, const float* normal, float4* plane, cudaStream_t s) {
	pm_pack_kernel<<<(n+255)/256, 256, 0, s>>>(n, depth, normal, plane);
	return cudaGetLastError();
}
cudaError_t pm_launch_unpack(int n, const float4* plane, float* depth, float* normal, cudaStream_t s) {
	pm_unpack_kernel<<<(n+255)/256, 256, 0, s>>>(n, plane, depth, normal);
	return cudaGetLastError();
}
