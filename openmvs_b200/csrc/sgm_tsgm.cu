// sgm_tsgm.cu — the per-level steps of the coarse-to-fine (tSGM) branch of SemiGlobalMatcher::Match(scene, ...)
// (libs/MVS/SemiGlobalMatcher.cpp:584-718) that surround the existing ragged match:
//   Disparity2RangeMap   per-pixel search ranges at twice the scale            SemiGlobalMatcher.cpp:1350-1444
//   FlipDirection        left->right map to a right->left map                  SemiGlobalMatcher.cpp:1630-1657
//   cv::filterSpeckles   small-region removal on int16 (OpenCV calib3d)        SemiGlobalMatcher.cpp:703-704
//   ExtractMask          border invalidation of the validity mask              SemiGlobalMatcher.cpp:1518-1575
//   UpscaleMask          mask to the next level's valid region                 SemiGlobalMatcher.cpp:1662-1690
//   cv::resize(INTER_AREA) of the 8-bit colour image                           SemiGlobalMatcher.h:127-142
// All integer arithmetic: every kernel is bit-exact with oracle/tsgm_oracle.cpp.
#include <cuda_runtime.h>
#include <cub/device/device_scan.cuh>
#include <stdint.h>

namespace {

constexpr int16_t NO_DISP = 32767;
constexpr int HW = 3;   // halfWindowSizeX/Y

// ---- Disparity2RangeMap ----
// One thread per coarse pixel; the 41x41 window of a NO_DISP pixel (most pixels of a sparse seed) and the 7x7 window of a
// valid one are read from a shared-memory tile (block + 20-pixel halo, NO_DISP outside the map).  GetMedian<Disparity>
// (libs/Common/List.h:668-678) is a selection by counting: a bisection over [min, max] for the (n/2)-th smallest value, and
// for an even count one more pass for the largest value below it.
constexpr int RB = 16, RHALO = 20, RT = RB+2*RHALO;

__device__ __forceinline__ int count_le(const int16_t (*t)[RT], int ty, int tx, int hw, int v) {
	int n = 0;
	for (int i = -hw; i <= hw; ++i) {
		const int16_t* row = t[ty+i];
		for (int j = -hw; j <= hw; ++j) { const int d = row[tx+j]; n += (d != NO_DISP && d <= v); }
	}
	return n;
}

__global__ void __launch_bounds__(RB*RB) range_coarse_kernel(const int16_t* __restrict__ D, int dw, int dh, const uint8_t* __restrict__ M, int mw,
	int minNumDisp, int minNumDispInvalid, uint32_t* __restrict__ range, int* __restrict__ maxNumDisp)
{
	__shared__ int16_t tile[RT][RT];
	const int x0 = blockIdx.x*RB-RHALO, y0 = blockIdx.y*RB-RHALO;
	for (int k = threadIdx.y*RB+threadIdx.x; k < RT*RT; k += RB*RB) {
		const int y = y0+k/RT, x = x0+k%RT;
		tile[k/RT][k%RT] = (x >= 0 && y >= 0 && x < dw && y < dh) ? D[(size_t)y*dw+x] : NO_DISP;
	}
	__syncthreads();
	const int c = blockIdx.x*RB+threadIdx.x, r = blockIdx.y*RB+threadIdx.y;
	int numDisp = 0;
	if (c < dw && r < dh) {
		int16_t minDisp = NO_DISP, maxDisp = NO_DISP;
		if (M[(size_t)(r*2+HW)*mw + c*2+HW] != 0) {
			const int ty = threadIdx.y+RHALO, tx = threadIdx.x+RHALO;
			const bool bInvalid = tile[ty][tx] == NO_DISP;
			const int hw = bInvalid ? 20 : 3;
			int n = 0, mn = 32767, mx = -32768;
			for (int i = -hw; i <= hw; ++i) for (int j = -hw; j <= hw; ++j) {
				const int d = tile[ty+i][tx+j];
				if (d != NO_DISP) { ++n; mn = min(mn, d); mx = max(mx, d); }
			}
			int16_t nd;
			if (n < 3) {
				maxDisp = (int16_t)min((int)(int16_t)(dw*2/3), minNumDispInvalid);
				minDisp = (int16_t)-maxDisp;
				nd = (int16_t)(maxDisp-minDisp);
			} else {
				// (n/2)-th smallest: the least v in [mn, mx] with count(<= v) > n/2
				const int k = n/2;
				int lo = mn, hi = mx;
				while (lo < hi) {
					const int mid = (lo+hi) >> 1;
					if (count_le(tile, ty, tx, hw, mid) > k) hi = mid; else lo = mid+1;
				}
				int med = lo;
				if (!(n & 1)) {
					int less = 0, below = -32768;
					for (int i = -hw; i <= hw; ++i) for (int j = -hw; j <= hw; ++j) {
						const int d = tile[ty+i][tx+j];
						if (d != NO_DISP && d < lo) { ++less; below = max(below, d); }
					}
					const int lower = less == k ? below : lo;
					med = (int16_t)((lower+lo)/2);
				}
				const int16_t disp = (int16_t)(med*2);
				nd = (int16_t)((mx-mn)*2);
				if (nd < minNumDisp) {
					nd = (int16_t)minNumDisp;
					minDisp = (int16_t)(disp-nd/2);
					maxDisp = (int16_t)(disp+(nd+1)/2);
				} else {
					const int16_t maxND = bInvalid ? 64 : 32;
					if (nd > maxND) {
						minDisp = (int16_t)(disp-(maxND*(disp-mn*2)+1)/nd);
						maxDisp = (int16_t)(disp+(maxND*(mx*2+1-disp)+1)/nd);
						nd = (int16_t)(maxDisp-minDisp);
					} else {
						minDisp = (int16_t)(disp-nd/2);
						maxDisp = (int16_t)(disp+(nd+1)/2);
					}
				}
			}
			numDisp = nd;
		}
		range[(size_t)r*dw+c] = (uint32_t)(uint16_t)minDisp | ((uint32_t)(uint16_t)maxDisp << 16);
	}
	numDisp = __reduce_max_sync(0xFFFFFFFFu, numDisp);
	if ((threadIdx.x & 31) == 0 && numDisp > 0) atomicMax(maxNumDisp, numDisp);
}

// the coarse pixel whose range fine pixel (y, x) receives: fine row 0 fills rows 0-4, coarse row r >= 1 rows 2r+3 and 2r+4, the last
// coarse row every remaining row; columns likewise (column 0 covers 5 columns, the tail copies its left neighbour)
__device__ __forceinline__ uint32_t fine_range(const uint32_t* range, int dw, int dh, int x, int y) {
	const int r = min(y < 5 ? 0 : (y-HW)/2, dh-1), c = min(x < 5 ? 0 : (x-HW)/2, dw-1);
	return range[(size_t)r*dw+c];
}
__device__ __forceinline__ int range_num(uint32_t v) { return (int16_t)((int)(int16_t)(v >> 16) - (int)(int16_t)(v & 0xFFFF)); }

__global__ void range_count_kernel(const uint32_t* __restrict__ range, int dw, int dh, int mw, int mh, unsigned long long* __restrict__ cnt) {
	const int x = blockIdx.x*blockDim.x+threadIdx.x, y = blockIdx.y*blockDim.y+threadIdx.y;
	if (x >= mw || y >= mh) return;
	cnt[(size_t)y*mw+x] = (unsigned long long)range_num(fine_range(range, dw, dh, x, y));
}

struct Pixel { unsigned long long idx; int16_t dmin, dmax; int pad; };

// the reference fills its pixel map row by row, so idx is the exclusive scan of the disparity counts in raster order
__global__ void range_write_kernel(const uint32_t* __restrict__ range, int dw, int dh, int mw, int mh, const unsigned long long* __restrict__ scan,
	Pixel* __restrict__ px, unsigned long long* __restrict__ total)
{
	const int x = blockIdx.x*blockDim.x+threadIdx.x, y = blockIdx.y*blockDim.y+threadIdx.y;
	if (x >= mw || y >= mh) return;
	const uint32_t v = fine_range(range, dw, dh, x, y);
	const size_t i = (size_t)y*mw+x;
	Pixel p; p.idx = scan[i]; p.dmin = (int16_t)(v & 0xFFFF); p.dmax = (int16_t)(v >> 16); p.pad = 0;
	px[i] = p;
	if (i+1 == (size_t)mw*mh) *total = scan[i] + (unsigned long long)range_num(v);
}

// ---- FlipDirection: the reference writes in raster order, so the LAST writer of a pixel (largest source column) wins: key =
// (column + 1) << 16 | -d, atomicMax per target pixel, 0 = never written (NO_DISP) ----
__global__ void flip_scatter_kernel(const int16_t* __restrict__ l2r, int w, int h, uint32_t* __restrict__ key) {
	const int c = blockIdx.x*blockDim.x+threadIdx.x, r = blockIdx.y;
	if (c >= w) return;
	const int d = l2r[(size_t)r*w+c];
	if (d == NO_DISP) return;
	const uint32_t k = ((uint32_t)(c+1) << 16) | (uint16_t)(int16_t)(-d);
	for (int x = max(c+d-1, 0), xe = min(c+d+2, w); x < xe; ++x)
		atomicMax(key+(size_t)r*w+x, k);
}
__global__ void flip_resolve_kernel(const uint32_t* __restrict__ key, int16_t* __restrict__ r2l, size_t n) {
	const size_t i = (size_t)blockIdx.x*blockDim.x+threadIdx.x;
	if (i >= n) return;
	const uint32_t k = key[i];
	r2l[i] = k ? (int16_t)(k & 0xFFFF) : NO_DISP;
}

// ---- cv::filterSpeckles: |a-b| <= maxDiff between two 4-neighbours that are not newVal is symmetric, so the regions are the
// connected components, found with the labelling of filter_kernels.cu (RemoveSmallSegments): link to the left (else upper)
// neighbour, pointer jumping, atomicMin unions over the upper edges the links did not take, pointer jumping again ----
__device__ __forceinline__ bool spk_edge(int a, int b, int newVal, int maxDiff) { return b != newVal && abs(a-b) <= maxDiff; }
__device__ __forceinline__ int spk_find(int* L, int i) {
	int p;
	while ((p = ((volatile int*)L)[i]) != i) i = p;
	return i;
}
__device__ void spk_union(int* L, int a, int b) {
	bool done;
	do {
		a = spk_find(L, a); b = spk_find(L, b);
		if (a < b) { const int old = atomicMin(L+b, a); done = (old == b); b = old; }
		else if (b < a) { const int old = atomicMin(L+a, b); done = (old == a); a = old; }
		else done = true;
	} while (!done);
}
__global__ void spk_init_kernel(const int16_t* __restrict__ img, int W, int H, int newVal, int maxDiff, int* L, int* size) {
	const int x = blockIdx.x*blockDim.x+threadIdx.x, y = blockIdx.y*blockDim.y+threadIdx.y;
	if (x >= W || y >= H) return;
	const int i = y*W+x;
	const int a = img[i];
	int l = -1;
	if (a != newVal) {
		l = i;
		if (x > 0 && spk_edge(a, img[i-1], newVal, maxDiff)) l = i-1;
		else if (y > 0 && spk_edge(a, img[i-W], newVal, maxDiff)) l = i-W;
	}
	L[i] = l;
	size[i] = 0;
}
__global__ void spk_jump_kernel(int* L, int n) {
	const int i = blockIdx.x*blockDim.x+threadIdx.x;
	if (i >= n) return;
	const int p = L[i];
	if (p >= 0 && p != i) L[i] = ((volatile int*)L)[p];
}
__global__ void spk_merge_kernel(const int16_t* __restrict__ img, int W, int H, int newVal, int maxDiff, int* L) {
	const int x = blockIdx.x*blockDim.x+threadIdx.x, y = blockIdx.y*blockDim.y+threadIdx.y;
	if (x < 1 || x >= W || y < 1 || y >= H) return;
	const int i = y*W+x;
	const int a = img[i];
	if (a == newVal) return;
	if (spk_edge(a, img[i-1], newVal, maxDiff) && spk_edge(a, img[i-W], newVal, maxDiff)) spk_union(L, i, i-W);
}
__global__ void spk_count_kernel(int* L, int* size, int n) {
	const int i = blockIdx.x*blockDim.x+threadIdx.x;
	int r = -1;
	if (i < n && L[i] >= 0) { r = spk_find(L, i); L[i] = r; }
	const unsigned peers = __match_any_sync(0xFFFFFFFFu, r);
	if (r >= 0 && (threadIdx.x&31) == __ffs(peers)-1) atomicAdd(size+r, __popc(peers));
}
__global__ void spk_remove_kernel(int16_t* __restrict__ img, const int* __restrict__ L, const int* __restrict__ size, int n, int newVal, int maxSize) {
	const int i = blockIdx.x*blockDim.x+threadIdx.x;
	if (i >= n) return;
	const int l = L[i];
	if (l >= 0 && size[l] <= maxSize) img[i] = (int16_t)newVal;
}

// ---- ExtractMask: one thread per row, the left-to-right pass, then the right-to-left pass over what it left ----
__global__ void extract_mask_kernel(const int16_t* __restrict__ disp, uint8_t* __restrict__ mask, int w, int h, int thValid) {
	const int r = blockIdx.x*blockDim.x+threadIdx.x;
	if (r >= h) return;
	const int16_t* d = disp + (size_t)r*w;
	uint8_t* m = mask + (size_t)r*w;
	int numValid = 0;
	for (int c = 0; c < w; ++c) {
		if (m[c] == 0) continue;
		m[c] = 0;
		if (d[c] == NO_DISP) continue;
		if (++numValid >= thValid) break;
	}
	numValid = 0;
	for (int c = w-1; c >= 0; --c) {
		if (m[c] == 0) continue;
		m[c] = 0;
		if (d[c] == NO_DISP) continue;
		if (++numValid >= thValid) break;
	}
}

// ---- UpscaleMask: fine (y, x) takes coarse ((y-3)/2, (x-3)/2) where that exists, else INVALID ----
__global__ void upscale_mask_kernel(const uint8_t* __restrict__ m, int w, int h, uint8_t* __restrict__ m2, int w2, int h2) {
	const int x = blockIdx.x*blockDim.x+threadIdx.x, y = blockIdx.y*blockDim.y+threadIdx.y;
	if (x >= w2 || y >= h2) return;
	const int r = (y-HW) >> 1, c = (x-HW) >> 1;
	m2[(size_t)y*w2+x] = (y >= HW && x >= HW && r < h && c < w) ? m[(size_t)r*w+c] : (uint8_t)0;
}

// ---- cv::resize(..., 1/f, 1/f, INTER_AREA) of an 8-bit image, integer f (OpenCV resizeAreaFast): a full f x f cell is
// (sum+2)>>2 for f = 2 (its vector path) and cvRound(sum*(1.f/(f*f))) otherwise; a cell cut by the border is cvRound((float)sum/count) ----
__global__ void resize_area_u8_kernel(const uint8_t* __restrict__ src, int sw, int sh, int ch, int f, uint8_t* __restrict__ dst, int dw, int dh) {
	const int x = blockIdx.x*blockDim.x+threadIdx.x, y = blockIdx.y*blockDim.y+threadIdx.y;
	if (x >= dw || y >= dh) return;
	const int sy0 = y*f, sx0 = x*f;
	const int ny = min(f, sh-sy0), nx = min(f, sw-sx0);
	const bool full = sy0+f <= sh && x < sw/f;
	const float scale = 1.f/(float)(f*f);
	for (int k = 0; k < ch; ++k) {
		int sum = 0;
		for (int j = 0; j < ny; ++j) {
			const uint8_t* row = src + ((size_t)(sy0+j)*sw + sx0)*ch + k;
			for (int i = 0; i < nx; ++i) sum += row[(size_t)i*ch];
		}
		int v;
		if (full) v = f == 2 ? (sum+2) >> 2 : __float2int_rn(__fmul_rn((float)sum, scale));
		else v = __float2int_rn(__fdiv_rn((float)sum, (float)(nx*ny)));
		dst[((size_t)y*dw+x)*ch+k] = (uint8_t)min(255, max(0, v));
	}
}

__global__ void fill_i16_kernel(int16_t* p, size_t n, int16_t v) {
	const size_t i = (size_t)blockIdx.x*blockDim.x+threadIdx.x;
	if (i < n) p[i] = v;
}

inline dim3 grid2(int w, int h, dim3 b) { return dim3((w+b.x-1)/b.x, (h+b.y-1)/b.y); }

} // namespace

// bytes of scratch the range map needs for an mw x mh pixel map: counts + scan (8 B each per pixel) + the CUB scan's temporary
size_t ts_range_scratch_bytes(int mw, int mh) {
	size_t tmp = 0;
	cub::DeviceScan::ExclusiveSum(nullptr, tmp, (const unsigned long long*)nullptr, (unsigned long long*)nullptr, mw*mh);
	return 16*(size_t)mw*mh + ((tmp+255) & ~(size_t)255);
}

// Disparity2RangeMap of D (dw x dh) over the fine valid region (mask mw x mh).  range: dw*dh words; scratch: ts_range_scratch_bytes;
// stat (device): [0] u64 numCosts, [1] low word = the largest disparity count.  Asynchronous; the caller reads stat back.
cudaError_t ts_launch_range_map(const int16_t* D, int dw, int dh, const uint8_t* M, int mw, int mh, int minNumDisp, int minNumDispInvalid,
	uint32_t* range, void* scratch, void* pixels, unsigned long long* stat, cudaStream_t s)
{
	cudaError_t e;
	if ((e = cudaMemsetAsync(stat, 0, 16, s)) != cudaSuccess) return e;
	range_coarse_kernel<<<grid2(dw, dh, dim3(RB, RB)), dim3(RB, RB), 0, s>>>(D, dw, dh, M, mw, minNumDisp, minNumDispInvalid, range, (int*)(stat+1));
	const size_t n = (size_t)mw*mh;
	unsigned long long* cnt = (unsigned long long*)scratch;
	unsigned long long* scan = cnt+n;
	void* tmp = scan+n;
	size_t tmpBytes = 0;
	cub::DeviceScan::ExclusiveSum(nullptr, tmpBytes, cnt, scan, (int)n);
	const dim3 b(32, 8);
	range_count_kernel<<<grid2(mw, mh, b), b, 0, s>>>(range, dw, dh, mw, mh, cnt);
	if ((e = cub::DeviceScan::ExclusiveSum(tmp, tmpBytes, cnt, scan, (int)n, s)) != cudaSuccess) return e;
	range_write_kernel<<<grid2(mw, mh, b), b, 0, s>>>(range, dw, dh, mw, mh, scan, (Pixel*)pixels, stat);
	return cudaGetLastError();
}
// key: w*h words of scratch
cudaError_t ts_launch_flip(const int16_t* l2r, int16_t* r2l, int w, int h, uint32_t* key, cudaStream_t s) {
	const size_t n = (size_t)w*h;
	cudaError_t e;
	if ((e = cudaMemsetAsync(key, 0, n*4, s)) != cudaSuccess) return e;
	flip_scatter_kernel<<<dim3((w+127)/128, h), 128, 0, s>>>(l2r, w, h, key);
	flip_resolve_kernel<<<(unsigned)((n+255)/256), 256, 0, s>>>(key, r2l, n);
	return cudaGetLastError();
}
// labels, sizes: w*h ints of scratch each
cudaError_t ts_launch_filter_speckles(int16_t* img, int w, int h, int newVal, int maxSize, int maxDiff, int* labels, int* sizes, cudaStream_t s) {
	const int n = w*h;
	const dim3 b(32, 8), g = grid2(w, h, b);
	spk_init_kernel<<<g, b, 0, s>>>(img, w, h, newVal, maxDiff, labels, sizes);
	int rounds = 1;
	while ((1<<rounds) < w+h) ++rounds;
	for (int r = 0; r < rounds; ++r) spk_jump_kernel<<<(n+255)/256, 256, 0, s>>>(labels, n);
	spk_merge_kernel<<<g, b, 0, s>>>(img, w, h, newVal, maxDiff, labels);
	for (int r = 0; r < rounds; ++r) spk_jump_kernel<<<(n+255)/256, 256, 0, s>>>(labels, n);
	spk_count_kernel<<<(n+255)/256, 256, 0, s>>>(labels, sizes, n);
	spk_remove_kernel<<<(n+255)/256, 256, 0, s>>>(img, labels, sizes, n, newVal, maxSize);
	return cudaGetLastError();
}
int ts_filter_speckles_launches(int w, int h) {
	int rounds = 1;
	while ((1<<rounds) < w+h) ++rounds;
	return 5+2*rounds;
}
cudaError_t ts_launch_extract_mask(const int16_t* disp, uint8_t* mask, int w, int h, int thValid, cudaStream_t s) {
	extract_mask_kernel<<<(h+63)/64, 64, 0, s>>>(disp, mask, w, h, thValid);
	return cudaGetLastError();
}
cudaError_t ts_launch_upscale_mask(const uint8_t* m, int w, int h, uint8_t* m2, int w2, int h2, cudaStream_t s) {
	const dim3 b(32, 8);
	upscale_mask_kernel<<<grid2(w2, h2, b), b, 0, s>>>(m, w, h, m2, w2, h2);
	return cudaGetLastError();
}
cudaError_t ts_launch_resize_area_u8(const uint8_t* src, int sw, int sh, int ch, int f, uint8_t* dst, int dw, int dh, cudaStream_t s) {
	const dim3 b(32, 8);
	resize_area_u8_kernel<<<grid2(dw, dh, b), b, 0, s>>>(src, sw, sh, ch, f, dst, dw, dh);
	return cudaGetLastError();
}
cudaError_t ts_launch_fill_i16(int16_t* p, size_t n, int16_t v, cudaStream_t s) {
	fill_i16_kernel<<<(unsigned)((n+255)/256), 256, 0, s>>>(p, n, v);
	return cudaGetLastError();
}
