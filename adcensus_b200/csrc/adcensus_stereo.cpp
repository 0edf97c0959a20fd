// adcensus_stereo.cpp -- the C++ drop-in class of include/ADCensusStereo.h, written purely on top of
// the C ABI (include/adcensus_b200.h).  Mirrors the call sequence and error truth table of the
// reference's ADCensusStereo (ADCensusStereo.cpp:21-67 Initialize, :69-132 Match, :134-144 Reset).
#include "../../include/ADCensusStereo.h"

#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "../../include/adcensus_b200.h"

static_assert(sizeof(ADCensusOption) == sizeof(adc_option), "option block must be byte-compatible with the C ABI");

ADCensusStereo::ADCensusStereo() : engine_(nullptr), width_(0), height_(0), max_disparity_range_(0), is_initialized_(false) {}

ADCensusStereo::~ADCensusStereo() {
    Release();
    is_initialized_ = false;
}

void ADCensusStereo::Release() {
    if (engine_) adc_destroy(engine_);
    engine_ = nullptr;
}

bool ADCensusStereo::Initialize(const sint32& width, const sint32& height, const ADCensusOption& option) {
    return Initialize(width, height, option, 0);
}

bool ADCensusStereo::Initialize(const sint32& width, const sint32& height, const ADCensusOption& option,
                                sint32 max_disparity_range) {
    width_ = width;
    height_ = height;
    option_ = option;
    max_disparity_range_ = max_disparity_range;
    Release();  // the reference leaks on a second Initialize; here the old engine is freed
    is_initialized_ = false;
    adc_option raw;
    std::memcpy(&raw, &option, sizeof(raw));
    adc_config cfg;
    std::memset(&cfg, 0, sizeof(cfg));
    if (const char* dev = std::getenv("ADC_B200_DEVICE")) cfg.device = std::atoi(dev);
    cfg.max_disparity_range = max_disparity_range;
    if (adc_create(width, height, &raw, &cfg, &engine_) != ADC_OK) {
        engine_ = nullptr;
        return false;
    }
    is_initialized_ = true;
    return true;
}

// The reference prints six timing lines from Match (ADCensusStereo.cpp:88-129); kept, with the
// device times of the corresponding stages, unless ADC_B200_QUIET is set.
static void print_stage_times(adc_engine* engine) {
    if (!std::getenv("ADC_B200_QUIET")) {
        float ms[6] = {0, 0, 0, 0, 0, 0};
        adc_last_stage_ms(engine, ms);
        std::printf("computing cost! timing :	%lf s\n", ms[0] / 1000.0);
        std::printf("cost aggregating! timing :	%lf s\n", ms[1] / 1000.0);
        std::printf("scanline optimizing! timing :	%lf s\n", ms[2] / 1000.0);
        std::printf("computing disparities! timing :	%lf s\n", ms[3] / 1000.0);
        std::printf("multistep refining! timing :	%lf s\n", ms[4] / 1000.0);
        std::printf("output disparities! timing :	%lf s\n", ms[5] / 1000.0);
    }
}

bool ADCensusStereo::Match(const uint8* img_left, const uint8* img_right, float32* disp_left) {
    if (!is_initialized_) return false;
    if (img_left == nullptr || img_right == nullptr || disp_left == nullptr) return false;
    if (adc_match(engine_, img_left, img_right, disp_left) != ADC_OK) return false;
    print_stage_times(engine_);
    return true;
}

bool ADCensusStereo::MatchWithConfidence(const uint8* img_left, const uint8* img_right, float32* disp_left, uint8* origin,
                                         float32* cost_best, float32* cost_second) {
    if (!is_initialized_) return false;
    if (img_left == nullptr || img_right == nullptr || disp_left == nullptr) return false;
    adc_aux_outputs aux = {origin, cost_best, cost_second, nullptr};
    if (adc_match_aux(engine_, img_left, img_right, disp_left, &aux) != ADC_OK) return false;
    print_stage_times(engine_);
    return true;
}

bool ADCensusStereo::Reset(const uint32& width, const uint32& height, const ADCensusOption& option) {
    Release();
    is_initialized_ = false;
    return Initialize(static_cast<sint32>(width), static_cast<sint32>(height), option, max_disparity_range_);
}

bool ADCensusStereo::MatchBatch(sint32 n, const uint8* left, const uint8* right, float32* disp) {
    if (!is_initialized_) return false;
    return adc_match_batch_strided(engine_, n, left, right, disp) == ADC_OK;
}
