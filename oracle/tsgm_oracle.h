/*
 * tsgm_oracle.h — C interface of the CPU oracle of the coarse-to-fine (tSGM) level loop (TEST INFRASTRUCTURE, not product code).
 * SemiGlobalMatcher::Match(scene, idxImage, numNeighbors, minResolution), libs/MVS/SemiGlobalMatcher.cpp:584-718.
 */
#ifndef B200MVS_TSGM_ORACLE_H_
#define B200MVS_TSGM_ORACLE_H_
#include "oracle.h"

#ifdef __cplusplus
extern "C" {
#endif

void oracle_sgm_tsgm_levels(int width, int height, int minResolution, int* nLevels, int* seedWidth, int* seedHeight);
/* cv::resize(..., 1./factor, 1./factor, INTER_AREA) of an 8-bit image with ch interleaved channels, integer factor */
void oracle_resize_area_u8(const uint8_t* src, int sw, int sh, int ch, int factor, uint8_t* dst);
uint64_t oracle_sgm_range_map(const int16_t* disparity, int dw, int dh, const uint8_t* mask, int mw, int mh,
	int minNumDisp, int minNumDispInvalid, oracle_sgm_pixel* pixels, int* maxNumDisp);
void oracle_sgm_flip_direction(const int16_t* l2r, int16_t* r2l, int width, int height);
void oracle_sgm_extract_mask(const int16_t* disparity, uint8_t* mask, int width, int height, int thValid);
void oracle_sgm_upscale_mask(const uint8_t* mask, int width, int height, uint8_t* mask2x, int w2, int h2);
void oracle_filter_speckles(int16_t* img, int width, int height, int newVal, int maxSpeckleSize, int maxDiff);
int oracle_sgm_match_tsgm(const float* leftGray, const uint8_t* leftBGR, const float* rightGray, const uint8_t* rightBGR,
	int width, int height, const uint8_t* leftMask, const uint8_t* rightMask, const int16_t* seed, int seedWidth, int seedHeight,
	int minResolution, int nSpeckleSize, int subpixelSteps, uint16_t P1, uint16_t P2, float P2alpha, float P2beta,
	int16_t* disparity, uint16_t* cost, uint64_t* levelCosts);

#ifdef __cplusplus
}
#endif
#endif
