/*
 * tsgm_oracle.cpp — CPU oracle of the coarse-to-fine (tSGM) level loop of SemiGlobalMatcher::Match(scene, ...)
 * (libs/MVS/SemiGlobalMatcher.cpp:584-718) for one rectified pair (TEST INFRASTRUCTURE ONLY, see oracle.h, tsgm_oracle.h).
 * The matches, cross-checks and the sub-pixel refinement are the oracle's own (sgm_oracle.cpp), the pyramid its cv::resize
 * restatements (pm_oracle.cpp); this file adds the steps between them.  Built with them into one library by tsgm_oracle.py.
 */
#include "tsgm_oracle.h"
#include <cmath>
#include <cstring>
#include <vector>
#include <algorithm>
#include <limits>

namespace {
constexpr int HW = 3;          // halfWindowSizeX/Y
constexpr int16_t NO_DISP = std::numeric_limits<int16_t>::max();
} // namespace

// ---- coarse-to-fine (tSGM) level loop of SemiGlobalMatcher::Match(scene, ...) (SemiGlobalMatcher.cpp:584-718) ----
namespace {

constexpr uint8_t MASK_INVALID = 0, MASK_VALID = 255;

// cv::saturate_cast<int>(double): round half to even
inline int saturate_round(double v) { return (int)std::nearbyint(v); }

// GetMedian<Disparity> (libs/Common/List.h:668-678): the middle element, or for an even count the two middle elements summed
// in int and divided by 2 (truncated toward zero), returned as Disparity
int16_t median_disparity(std::vector<int16_t> v) {
	std::sort(v.begin(), v.end());
	const size_t n = v.size();
	if (n % 2) return v[n/2];
	return (int16_t)(((int)v[n/2-1] + (int)v[n/2]) / 2);
}

} // namespace

extern "C" {

// computeMaxResolution (libs/Common/Types.inl:2459-2477) with level = 8, then the scale of SemiGlobalMatcher.cpp:584-589 and the
// seed size of :620-624 (computeResize of the coarsest level by 0.5, Types.inl:2440-2445, minus the 3-pixel border)
void oracle_sgm_tsgm_levels(int width, int height, int minResolution, int* nLevels, int* seedWidth, int* seedHeight) {
	const unsigned imageSize = (unsigned)std::max(width, height);
	unsigned level = 8;
	if ((imageSize >> level) < (unsigned)minResolution) {
		level = 0;
		while ((imageSize >> (level+1)) >= (unsigned)minResolution)
			++level;
	}
	const int L = std::max(1u, level);   // scale = 1/max(2, 2^level)
	*nLevels = L+1;
	const double scale = 1.0/(double)(1u << L);
	const int cw = saturate_round(width*scale), ch = saturate_round(height*scale);
	*seedWidth = saturate_round(cw*0.5)-2*HW;
	*seedHeight = saturate_round(ch*0.5)-2*HW;
}

// cv::resize(src, dst, Size(), 1./factor, 1./factor, INTER_AREA) of an 8-bit image with `ch` interleaved channels and an
// integer factor (OpenCV's resizeAreaFast: full cells of factor 2 are (sum+2)>>2, other full cells cvRound(sum*(1.f/area)),
// cells cut by the image border cvRound((float)sum/count)); dst is computeResize(size, 1./factor)
void oracle_resize_area_u8(const uint8_t* src, int sw, int sh, int ch, int factor, uint8_t* dst) {
	const int dw = saturate_round(sw*(1.0/factor)), dh = saturate_round(sh*(1.0/factor));
	const int fullW = sw/factor;
	const float scale = 1.f/(float)(factor*factor);
	for (int y=0; y<dh; ++y) for (int x=0; x<dw; ++x) for (int k=0; k<ch; ++k) {
		const int sy0 = y*factor, sx0 = x*factor;
		int sum = 0, count = 0;
		for (int j=0; j<factor && sy0+j<sh; ++j)
			for (int i=0; i<factor && sx0+i<sw; ++i) { sum += src[((size_t)(sy0+j)*sw+sx0+i)*ch+k]; ++count; }
		int v;
		if (sy0+factor <= sh && x < fullW) v = factor == 2 ? (sum+2)>>2 : (int)std::nearbyint((float)sum*scale);
		else v = (int)std::nearbyint((float)sum/(float)count);
		dst[((size_t)y*dw+x)*ch+k] = (uint8_t)std::min(255, std::max(0, v));
	}
}

// Disparity2RangeMap (SemiGlobalMatcher.cpp:1350-1444): per-pixel search ranges at twice the scale of `disparity` (dw x dh)
// over the valid region of the finer level (mask, mw x mh); pixels receives mw x mh records.  Returns numCosts.
uint64_t oracle_sgm_range_map(const int16_t* disparity, int dw, int dh, const uint8_t* mask, int mw, int mh,
	int minNumDisp, int minNumDispInvalid, oracle_sgm_pixel* pixels, int* maxNumDispOut)
{
	uint64_t numCosts = 0;
	int maxNumDisp = 0;
	std::vector<int16_t> disps;
	auto D = [&](int r, int c) { return disparity[(size_t)r*dw+c]; };
	for (int r=0; r<dh; ++r) {
		const int r2 = r == 0 ? 0 : r*2+HW;
		const int offset = r2*mw;
		int c2e = HW;
		const uint8_t* pm = mask + (size_t)(r*2+HW)*mw + HW;
		for (int c=0, c2=0; c<dw; ++c, pm+=2) {
			int16_t numDisp, minDisp, maxDisp;
			if (*pm == MASK_INVALID) {
				minDisp = maxDisp = NO_DISP;
				numDisp = 0;
			} else {
				const bool bInvalid = D(r,c) == NO_DISP;
				disps.clear();
				const int hw = bInvalid ? 20 : 3;
				for (int i=-hw; i<=hw; ++i) for (int j=-hw; j<=hw; ++j) {
					const int x = c+j, y = r+i;
					if (x >= 0 && y >= 0 && x < dw && y < dh && D(y,x) != NO_DISP)
						disps.push_back(D(y,x));
				}
				if (disps.size() < 3) {
					maxDisp = std::min((int16_t)(dw*2/3), (int16_t)minNumDispInvalid);
					minDisp = (int16_t)-maxDisp;
					numDisp = (int16_t)(maxDisp-minDisp);
				} else {
					const int16_t disp = (int16_t)(median_disparity(disps)*2);
					const int16_t mn = *std::min_element(disps.begin(), disps.end()), mx = *std::max_element(disps.begin(), disps.end());
					numDisp = (int16_t)((mx-mn)*2);
					if (numDisp < minNumDisp) {
						numDisp = (int16_t)minNumDisp;
						minDisp = (int16_t)(disp-numDisp/2);
						maxDisp = (int16_t)(disp+(numDisp+1)/2);
					} else {
						const int16_t maxND = bInvalid ? 64 : 32;
						if (numDisp > maxND) {
							minDisp = (int16_t)(disp-(maxND*(disp-mn*2)+1)/numDisp);
							maxDisp = (int16_t)(disp+(maxND*(mx*2+1-disp)+1)/numDisp);
							numDisp = (int16_t)(maxDisp-minDisp);
						} else {
							minDisp = (int16_t)(disp-numDisp/2);
							maxDisp = (int16_t)(disp+(numDisp+1)/2);
						}
					}
				}
				maxNumDisp = std::max(maxNumDisp, (int)numDisp);
			}
			c2e += 2;
			do {
				oracle_sgm_pixel& p = pixels[offset+c2];
				p.dmin = minDisp; p.dmax = maxDisp; p.idx = numCosts; p.reserved = 0;
				numCosts += numDisp;
			} while (++c2 < c2e);
		}
		do {
			const oracle_sgm_pixel& p = pixels[offset+c2e-1];
			oracle_sgm_pixel& q = pixels[offset+c2e];
			q.dmin = p.dmin; q.dmax = p.dmax; q.idx = numCosts; q.reserved = 0;
			numCosts += (int16_t)(p.dmax-p.dmin);
		} while (++c2e < mw);
		const int offsete = (r+1 == dh ? mh : r*2+HW+2)*mw;
		for (int o=offset+mw; o<offsete; o+=mw) for (int c2=0; c2<mw; ++c2) {
			const oracle_sgm_pixel& p = pixels[offset+c2];
			oracle_sgm_pixel& q = pixels[o+c2];
			q.dmin = p.dmin; q.dmax = p.dmax; q.idx = numCosts; q.reserved = 0;
			numCosts += (int16_t)(p.dmax-p.dmin);
		}
	}
	if (maxNumDispOut) *maxNumDispOut = maxNumDisp;
	return numCosts;
}

// FlipDirection (SemiGlobalMatcher.cpp:1630-1657): r2l (same size) = NO_DISP, then every valid d writes -d to 3 pixels in raster order
void oracle_sgm_flip_direction(const int16_t* l2r, int16_t* r2l, int width, int height) {
	for (size_t i=0, n=(size_t)width*height; i<n; ++i) r2l[i] = NO_DISP;
	for (int r=0; r<height; ++r) for (int c=0; c<width; ++c) {
		const int16_t d = l2r[(size_t)r*width+c];
		if (d == NO_DISP) continue;
		for (int x=std::max(c+d-1, 0), xe=std::min(c+d+2, width); x<xe; ++x)
			r2l[(size_t)r*width+x] = (int16_t)-d;
	}
}

// ExtractMask (SemiGlobalMatcher.cpp:1518-1575): per row a left-to-right pass, then a right-to-left pass; each invalidates the
// mask up to and including the thValid-th valid disparity it meets
void oracle_sgm_extract_mask(const int16_t* disparity, uint8_t* mask, int width, int height, int thValid) {
	for (int pass=0; pass<2; ++pass) for (int r=0; r<height; ++r) {
		int numValid = 0;
		for (int k=0; k<width; ++k) {
			const int c = pass == 0 ? k : width-1-k;
			uint8_t& m = mask[(size_t)r*width+c];
			if (m == MASK_INVALID) continue;
			m = MASK_INVALID;
			if (disparity[(size_t)r*width+c] == NO_DISP) continue;
			if (++numValid >= thValid) break;
		}
	}
}

// UpscaleMask (SemiGlobalMatcher.cpp:1662-1690): mask2x (w2 x h2) = INVALID, coarse (r,c) -> the 2x2 cell at (2r+3, 2c+3)
void oracle_sgm_upscale_mask(const uint8_t* mask, int width, int height, uint8_t* mask2x, int w2, int h2) {
	memset(mask2x, MASK_INVALID, (size_t)w2*h2);
	for (int r=0; r<height; ++r) for (int c=0; c<width; ++c)
		for (int i=0; i<2; ++i) for (int j=0; j<2; ++j) {
			const int y = r*2+HW+i, x = c*2+HW+j;
			if (x < w2 && y < h2) mask2x[(size_t)y*w2+x] = mask[(size_t)r*width+c];
		}
}

// cv::filterSpeckles(img, newVal, maxSpeckleSize, maxDiff) on int16 (OpenCV calib3d, filterSpecklesImpl): 4-connected regions
// of values != newVal whose neighbours differ by <= maxDiff; regions of at most maxSpeckleSize pixels become newVal
void oracle_filter_speckles(int16_t* img, int width, int height, int newVal, int maxSpeckleSize, int maxDiff) {
	const size_t n = (size_t)width*height;
	std::vector<int> labels(n, 0);
	std::vector<uint8_t> rtype(1, 0);
	std::vector<int> stack;
	int curlabel = 0;
	for (int i=0; i<height; ++i) for (int j=0; j<width; ++j) {
		const size_t p0 = (size_t)i*width+j;
		if (img[p0] == newVal) continue;
		if (labels[p0]) {
			if (rtype[labels[p0]]) img[p0] = (int16_t)newVal;
			continue;
		}
		labels[p0] = ++curlabel;
		int count = 0;
		stack.assign(1, (int)p0);
		while (!stack.empty()) {
			const int p = stack.back(); stack.pop_back();
			++count;
			const int y = p/width, x = p%width;
			const int dp = img[p];
			auto push = [&](int q) {
				if (!labels[q] && img[q] != newVal && std::abs(dp-(int)img[q]) <= maxDiff) { labels[q] = curlabel; stack.push_back(q); }
			};
			if (y < height-1) push(p+width);
			if (y > 0) push(p-width);
			if (x < width-1) push(p+1);
			if (x > 0) push(p-1);
		}
		rtype.push_back(count <= maxSpeckleSize ? 1 : 0);
		if (rtype[curlabel]) img[p0] = (int16_t)newVal;
	}
}

// the level loop of SemiGlobalMatcher::Match(scene, ...) (SemiGlobalMatcher.cpp:584-718) for one rectified pair: full-resolution
// gray / BGR images, masks (nullable: all valid), seed (nullable: all NO_DISP; seedWidth x seedHeight from oracle_sgm_tsgm_levels).
// disparity / cost receive the refined left disparity (x subpixelSteps) and the cost map of the last left match over the
// (width-6) x (height-6) valid region; levelCosts (nullable, 2 per level) the size of the right and the left cost volume of every
// level.  Returns 0, or 1 on a size mismatch.
int oracle_sgm_match_tsgm(const float* leftGray, const uint8_t* leftBGR, const float* rightGray, const uint8_t* rightBGR,
	int width, int height, const uint8_t* leftMask, const uint8_t* rightMask, const int16_t* seed, int seedWidth, int seedHeight,
	int minResolution, int nSpeckleSize, int subpixelSteps, uint16_t P1, uint16_t P2, float P2alpha, float P2beta,
	int16_t* disparity, uint16_t* cost, uint64_t* levelCosts)
{
	int nLevels, sw, sh;
	oracle_sgm_tsgm_levels(width, height, minResolution, &nLevels, &sw, &sh);
	if (seed && (seedWidth != sw || seedHeight != sh)) return 1;
	if (sw <= 0 || sh <= 0) return 1;
	std::vector<int16_t> leftD(seed ? seed : (const int16_t*)nullptr, seed ? seed+(size_t)sw*sh : (const int16_t*)nullptr), rightD;
	if (!seed) leftD.assign((size_t)sw*sh, NO_DISP);
	int pw = sw, ph = sh;   // size of the disparity maps of the previous level
	std::vector<uint8_t> leftM, rightM;
	std::vector<oracle_sgm_pixel> px;
	std::vector<uint8_t> costs; std::vector<uint16_t> accums;
	std::vector<int16_t> rDisp;
	std::vector<uint16_t> lCost;
	for (int level=0; level<nLevels; ++level) {
		const int factor = 1 << (nLevels-1-level);
		const bool first = level == 0;
		// ViewData::GetImage(scale) (SemiGlobalMatcher.h:127-142)
		int lw = width, lh = height;
		std::vector<float> lg, rg; std::vector<uint8_t> lc, rc;
		const float *LG = leftGray, *RG = rightGray; const uint8_t *LC = leftBGR, *RC = rightBGR;
		if (factor > 1) {
			lw = saturate_round(width*(1.0/factor)); lh = saturate_round(height*(1.0/factor));
			lg.resize((size_t)lw*lh); rg.resize((size_t)lw*lh); lc.resize((size_t)lw*lh*3); rc.resize((size_t)lw*lh*3);
			oracle_resize_area(leftGray, width, height, lg.data(), lw, lh, factor, factor);
			oracle_resize_area(rightGray, width, height, rg.data(), lw, lh, factor, factor);
			oracle_resize_area_u8(leftBGR, width, height, 3, factor, lc.data());
			oracle_resize_area_u8(rightBGR, width, height, 3, factor, rc.data());
			LG = lg.data(); RG = rg.data(); LC = lc.data(); RC = rc.data();
		}
		const int vw = lw-2*HW, vh = lh-2*HW;
		if (vw <= 0 || vh <= 0) return 1;
		if (first) {
			// masks: NEAREST to the level size, then the valid ROI (:626-631)
			for (int m=0; m<2; ++m) {
				const uint8_t* src = m == 0 ? leftMask : rightMask;
				std::vector<uint8_t>& dst = m == 0 ? leftM : rightM;
				dst.assign((size_t)vw*vh, MASK_VALID);
				if (!src) continue;
				std::vector<float> f((size_t)width*height), g((size_t)lw*lh);
				for (size_t i=0; i<f.size(); ++i) f[i] = src[i];
				oracle_resize_nearest(f.data(), width, height, 1, g.data(), lw, lh);
				for (int r=0; r<vh; ++r) for (int c=0; c<vw; ++c) dst[(size_t)r*vw+c] = (uint8_t)g[(size_t)(r+HW)*lw+c+HW];
			}
		} else {
			for (int m=0; m<2; ++m) {
				std::vector<uint8_t>& M = m == 0 ? leftM : rightM;
				std::vector<uint8_t> up((size_t)vw*vh);
				oracle_sgm_upscale_mask(M.data(), pw, ph, up.data(), vw, vh);
				M.swap(up);
			}
		}
		const int minND = first ? 11 : 5, minNDI = first ? 33 : 7;
		px.resize((size_t)vw*vh);
		// right -> left (:641-642, 672)
		rightD.resize((size_t)pw*ph);
		oracle_sgm_flip_direction(leftD.data(), rightD.data(), pw, ph);
		uint64_t numCosts = oracle_sgm_range_map(rightD.data(), pw, ph, rightM.data(), vw, vh, minND, minNDI, px.data(), nullptr);
		if (levelCosts) levelCosts[2*level] = numCosts;
		costs.assign(numCosts, 0); accums.assign(numCosts, 0);
		rDisp.resize((size_t)vw*vh); lCost.resize((size_t)vw*vh);
		oracle_sgm_match(RG, RC, LG, lw, lh, px.data(), numCosts, P1, P2, P2alpha, P2beta, 3, costs.data(), accums.data(), rDisp.data(), lCost.data());
		// left -> right (:675-685)
		numCosts = oracle_sgm_range_map(leftD.data(), pw, ph, leftM.data(), vw, vh, minND, minNDI, px.data(), nullptr);
		if (levelCosts) levelCosts[2*level+1] = numCosts;
		costs.assign(numCosts, 0); accums.assign(numCosts, 0);
		leftD.resize((size_t)vw*vh);
		oracle_sgm_match(LG, LC, RG, lw, lh, px.data(), numCosts, P1, P2, P2alpha, P2beta, 3, costs.data(), accums.data(), leftD.data(), lCost.data());
		if (first) {
			// :698-706, in sequence: the right map is checked against the already-checked left map
			oracle_sgm_cross_check(leftD.data(), rDisp.data(), vw, vh, 1);
			oracle_sgm_cross_check(rDisp.data(), leftD.data(), vw, vh, 1);
			oracle_filter_speckles(leftD.data(), vw, vh, NO_DISP, nSpeckleSize, 5);
			oracle_filter_speckles(rDisp.data(), vw, vh, NO_DISP, nSpeckleSize, 5);
			oracle_sgm_extract_mask(leftD.data(), leftM.data(), vw, vh, 3);
			oracle_sgm_extract_mask(rDisp.data(), rightM.data(), vw, vh, 3);
		} else {
			oracle_sgm_cross_check(leftD.data(), rDisp.data(), vw, vh, 1);
		}
		pw = vw; ph = vh;
	}
	// RefineDisparityMap with the pixel map and accumulated costs of the last left match (:718)
	oracle_sgm_refine(px.data(), accums.data(), leftD.data(), pw*ph, subpixelSteps);
	if (pw != width-2*HW || ph != height-2*HW) return 1;
	memcpy(disparity, leftD.data(), sizeof(int16_t)*pw*ph);
	memcpy(cost, lCost.data(), sizeof(uint16_t)*pw*ph);
	return 0;
}

} // extern "C"
