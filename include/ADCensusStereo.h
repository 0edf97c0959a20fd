// include/ADCensusStereo.h -- header-compatible shim of the reference's ADCensusStereo class
// (reference ADCensusStereo.h:14-95).  Same class name and the same three public methods with
// the same signatures, error behaviour (bool) and buffer contracts; the four by-value CPU stage
// objects of the reference are replaced by one opaque handle into the CUDA engine.
//
//   ADCensusStereo stereo;                       // main.cpp:97
//   stereo.Initialize(width, height, option);    // main.cpp:103
//   stereo.Match(bgr_left, bgr_right, disparity);// main.cpp:118
//
// Link with libadcensus_b200.so.  Everything runs on the GPU; there is no CPU fallback: if no
// usable device is present Initialize returns false and adc_last_error() says why.
#ifndef ADCENSUS_B200_STEREO_H_
#define ADCENSUS_B200_STEREO_H_

#include "adcensus_types.h"

struct adc_engine;

class ADCensusStereo {
public:
    ADCensusStereo();
    ~ADCensusStereo();
    ADCensusStereo(const ADCensusStereo&) = delete;
    ADCensusStereo& operator=(const ADCensusStereo&) = delete;

    // Allocates the device arena for width x height x (max-min disparity).  false when
    // width<=0, height<=0 or the disparity range is empty (reference ADCensusStereo.cpp:31,38),
    // or when the CUDA engine cannot be created.
    bool Initialize(const sint32& width, const sint32& height, const ADCensusOption& option);

    // img_left/img_right: packed BGR u8, row stride 3*width; disp_left: width*height float32,
    // Invalid_Float marks invalid pixels.  false before Initialize or on a null pointer
    // (reference ADCensusStereo.cpp:71-76).
    bool Match(const uint8* img_left, const uint8* img_right, float32* disp_left);

    // Release + Initialize (reference ADCensusStereo.cpp:134-144).
    bool Reset(const uint32& width, const uint32& height, const ADCensusOption& option);

    // ---- extensions (not in the reference) ----
    // Initialize with this object's disparity range limit set (adc_config.max_disparity_range: 0 = the default
    // ADC_MAX_DISPARITY_RANGE, at most ADC_MAX_DISPARITY_RANGE_WIDE); Reset keeps the limit.  The three-argument
    // Initialize uses the default limit.
    bool Initialize(const sint32& width, const sint32& height, const ADCensusOption& option, sint32 max_disparity_range);
    // n independent pairs in one call: left/right [n][H][W][3], disp [n][H][W] (host memory).
    bool MatchBatch(sint32 n, const uint8* left, const uint8* right, float32* disp);
    // Match plus per-pixel confidence (adc_match_aux): origin = ADC_ORIGIN_* code of each pixel (measured, voted,
    // interpolated, invalid), cost_best / cost_second = the winner's aggregated cost and the least cost two or more
    // disparities away from it.  width*height each; any of the three may be null.  Prints the timing lines Match prints.
    bool MatchWithConfidence(const uint8* img_left, const uint8* img_right, float32* disp_left, uint8* origin,
                             float32* cost_best, float32* cost_second);
    adc_engine* handle() const { return engine_; }

private:
    void Release();
    adc_engine* engine_;
    sint32 width_, height_;
    ADCensusOption option_;
    sint32 max_disparity_range_;
    bool is_initialized_;
};

#endif
