/* include/adcensus_b200.h -- the drop-in boundary of the B200-native AD-Census engine.
 *
 * A plain C ABI (extern "C", raw pointers and sizes, no torch / CUDA types) over the sm_100a
 * kernels in adcensus_b200/csrc.  The reference (ethan-li-coding/AD-Census) has no FFI of its
 * own: its boundary is the C++ class ADCensusStereo (ADCensusStereo.h:14-95) compiled into the
 * caller.  include/ADCensusStereo.h in this repo is the header-compatible shim of that class and
 * is implemented purely in terms of the functions declared here; INTEGRATION.md shows how an
 * existing caller of the reference switches over.
 *
 * Each entry point names the reference interface it stands in for.
 */
#ifndef ADCENSUS_B200_H_
#define ADCENSUS_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Byte-identical to the reference's ADCensusOption (adcensus_types.h:45-75): 60 bytes, align 4.
 * A pointer to the reference's struct may be passed wherever adc_option is expected. */
typedef struct adc_option {
    int32_t min_disparity;   /* offset  0 */
    int32_t max_disparity;   /*         4   (exclusive) */
    int32_t lambda_ad;       /*         8 */
    int32_t lambda_census;   /*        12 */
    int32_t cross_L1;        /*        16 */
    int32_t cross_L2;        /*        20 */
    int32_t cross_t1;        /*        24 */
    int32_t cross_t2;        /*        28 */
    float   so_p1;           /*        32 */
    float   so_p2;           /*        36 */
    int32_t so_tso;          /*        40 */
    int32_t irv_ts;          /*        44 */
    float   irv_th;          /*        48 */
    float   lrcheck_thres;   /*        52 */
    uint8_t do_lr_check;     /*        56   (C++ bool in the reference) */
    uint8_t do_filling;      /*        57 */
    uint8_t do_discontinuity_adjustment; /* 58 */
    uint8_t reserved_;       /*        59   padding byte, ignored */
} adc_option;

typedef struct adc_engine adc_engine; /* opaque; owns the device arena, streams and tables */

/* error codes (0 = success).  adc_last_error() gives the text for the calling thread. */
enum {
    ADC_OK = 0,
    ADC_ERR_ARG = 1,          /* null pointer / non-positive size / empty disparity range: the cases where
                                 the reference's Initialize/Match return false (ADCensusStereo.cpp:31,38,71,74) */
    ADC_ERR_CUDA = 2,         /* a CUDA runtime call failed */
    ADC_ERR_UNSUPPORTED = 3,  /* configuration outside what the kernels implement (see DESIGN.md) */
    ADC_ERR_NOMEM = 4         /* device or pinned-host allocation failed */
};

/* Engine tuning knobs; zero-initialise for defaults. */
typedef struct adc_config {
    int32_t device;          /* CUDA device ordinal */
    int32_t wave_pairs;      /* stereo pairs processed by one batched kernel launch (default: auto) */
    int32_t lanes;           /* concurrent waves in flight, one stream each (default: auto) */
    int32_t debug_flags;     /* test hooks, 0 in production: force the alternate code paths that otherwise only unusual
                                parameters reach, so that the parity tests can run every shipped kernel (ADC_DBG_*) */
    int32_t max_disparity_range; /* offset 16: largest max_disparity - min_disparity this engine accepts.  0 =
                                ADC_MAX_DISPARITY_RANGE; 1 .. ADC_MAX_DISPARITY_RANGE_WIDE raise (or lower) it; anything
                                else fails adc_create with ADC_ERR_ARG.  adc_get_config reports the resolved value. */
    int32_t reserved[11];    /* must be zero */
} adc_config;

enum {
    ADC_DBG_NO_RAY_TABLE = 1,     /* interpolation evaluates lround(y + m*sin) in double per step instead of the verified integer table */
    ADC_DBG_VOTE_ENUM = 2,        /* region voting finds the affected histograms by enumeration instead of adjacency lists */
    ADC_DBG_VOTE_GLOBAL_STATE = 4,/* region voting keeps its per-slot state in global instead of shared memory */
    ADC_DBG_UNFUSED_AGG = 8       /* aggregation as eight single passes instead of five (three of them fused double passes) */
};

/* stands in for: ADCensusOption::ADCensusOption() defaults (adcensus_types.h:67-74) */
void adc_default_option(adc_option* opt);

/* Sizes the kernels implement; the reference has no such limits (it only rejects non-positive sizes).  A configuration
 * outside them fails at adc_create / Initialize with ADC_ERR_UNSUPPORTED -- never later, in adc_match.
 * The disparity range limit is per engine: ADC_MAX_DISPARITY_RANGE unless adc_config.max_disparity_range sets another
 * value, at most ADC_MAX_DISPARITY_RANGE_WIDE (the scanline kernel keeps up to 16 disparities per lane of a warp). */
#define ADC_MAX_DISPARITY_RANGE 256        /* max_disparity - min_disparity, default limit */
#define ADC_MAX_DISPARITY_RANGE_WIDE 512   /* largest limit adc_config.max_disparity_range may set */
#define ADC_MAX_HEIGHT 4096
#define ADC_MAX_WIDTH 10000           /* also bounds width + disparity range */

/* stands in for: ADCensusStereo::Initialize(width, height, option) (ADCensusStereo.h:25,
 * ADCensusStereo.cpp:21-67).  cfg may be NULL.  Fails (ADC_ERR_ARG) exactly where Initialize
 * returns false: width<=0, height<=0, max_disparity-min_disparity<=0, and on a cfg->max_disparity_range outside
 * 0 .. ADC_MAX_DISPARITY_RANGE_WIDE; fails with ADC_ERR_UNSUPPORTED beyond the limits above. */
int adc_create(int32_t width, int32_t height, const adc_option* opt, const adc_config* cfg, adc_engine** out);

/* stands in for: ADCensusStereo::~ADCensusStereo / Release (ADCensusStereo.cpp:15-19,312-316) */
void adc_destroy(adc_engine* e);

/* stands in for: ADCensusStereo::Match(img_left, img_right, disp_left) (ADCensusStereo.h:33,
 * ADCensusStereo.cpp:69-132).  Packed BGR u8 [H][W][3] host images (main.cpp:61-76), caller-
 * allocated float32 [H][W] host output, +inf = invalid.  Synchronous. */
int adc_match(adc_engine* e, const uint8_t* img_left, const uint8_t* img_right, float* disp_left);

/* The right-view disparity map of the most recent adc_match call: what the reference computes into its private
 * disp_right_ (ADCensusStereo::ComputeDisparityRight, ADCensusStereo.cpp:245-310) for the left-right check and never
 * hands out -- float32 [H][W], sub-pixel, not refined (a minimum at either end of the range is the integer disparity).
 * Host pointer.  SURVEY.md 8(f) rank 4.  Batch callers get the same map per pair through adc_aux_outputs.disp_right of
 * adc_match_batch_strided_aux / adc_match_batch_device_aux. */
int adc_get_right_disparity(adc_engine* e, float* disp_right);

/* ---- side outputs (confidence) ----------------------------------------------------------------
 * Per pair, [H][W], left view, of the same run as the map they come with:
 *   origin       how the pixel's value was obtained, before discontinuity adjustment and the median filter (those two
 *                stages touch every pixel and do not change it): one ADC_ORIGIN_* code, with ADC_ORIGIN_WTA_INVALID
 *                OR-ed on where WTA itself returned Invalid_Float (the minimum lay at an end of the disparity range).
 *   cost_best    min over d in [0, D) of the aggregated cost WTA scans (the output of the fourth scanline pass): the
 *                cost of the WTA winner b (the first minimum in ascending d).
 *   cost_second  min of that cost over the d with |d - b| >= 2; +inf where there is none (range < 3, or range 3 with
 *                b = 1).  cost_best / cost_second is the usual peak-ratio confidence.
 *   disp_right   the right-view map, exactly what adc_get_right_disparity returns after adc_match of that pair.
 * Any member may be NULL (not wanted).  aux == NULL, or all four members NULL, runs exactly the plain call. */
typedef struct adc_aux_outputs {
    uint8_t* origin;      /* [n][H][W] ADC_ORIGIN_* */
    float*   cost_best;   /* [n][H][W] */
    float*   cost_second; /* [n][H][W] */
    float*   disp_right;  /* [n][H][W] */
} adc_aux_outputs;

enum {
    ADC_ORIGIN_MATCHED = 0,            /* a WTA value that passed the left-right check (any finite WTA value without it) */
    ADC_ORIGIN_VOTED_MISMATCH = 1,     /* in the mismatch list after the outlier stage, filled by region voting */
    ADC_ORIGIN_VOTED_OCCLUSION = 2,    /* in the occlusion list after the outlier stage, filled by region voting */
    ADC_ORIGIN_INTERP_MISMATCH = 3,    /* still in the mismatch list after voting, filled by proper interpolation */
    ADC_ORIGIN_INTERP_OCCLUSION = 4,   /* still in the occlusion list after voting, filled by proper interpolation */
    ADC_ORIGIN_INVALID = 5,            /* still Invalid_Float after the last filling step that ran */
    ADC_ORIGIN_WTA_INVALID = 8         /* flag: WTA returned Invalid_Float (minimum at an end of the range) */
};

/* adc_match with side outputs.  Host pointers, synchronous.  The side outputs' device scratch and pinned staging are
 * allocated on the first call that asks for them (ADC_ERR_NOMEM if that fails; the engine stays usable). */
int adc_match_aux(adc_engine* e, const uint8_t* img_left, const uint8_t* img_right, float* disp_left,
                  const adc_aux_outputs* aux);

/* Batched Match over n independent pairs (the data-parallel form of the call above; the
 * reference would loop Match).  Pointers are host pointers; pinned buffers are copied
 * asynchronously straight from/to the caller's memory, pageable ones go through an internal
 * pinned staging ring.  Synchronous: returns when every disp_left[i] is complete. */
int adc_match_batch(adc_engine* e, int32_t n, const uint8_t* const* img_left,
                    const uint8_t* const* img_right, float* const* disp_left);

/* Same, contiguous host arrays: left/right [n][H][W][3], disp [n][H][W]. */
int adc_match_batch_strided(adc_engine* e, int32_t n, const uint8_t* left, const uint8_t* right, float* disp);
/* Same, with side outputs (see adc_aux_outputs): host buffers, pageable or pinned, synchronous. */
int adc_match_batch_strided_aux(adc_engine* e, int32_t n, const uint8_t* left, const uint8_t* right, float* disp,
                                const adc_aux_outputs* aux);

/* Same, but the arrays already live in device memory (HBM-resident form used for the
 * kernel-only throughput figure).  Work is enqueued on the engine's streams, fork/joined on
 * `stream` (a cudaStream_t passed as void*, NULL = legacy default stream) and NOT synchronised:
 * the caller brackets it with its own events. */
int adc_match_batch_device(adc_engine* e, int32_t n, const uint8_t* d_left, const uint8_t* d_right,
                           float* d_disp, void* stream);
/* Same, with side outputs (see adc_aux_outputs) in device memory, complete when d_disp is (in pipelined mode: after
 * adc_join). */
int adc_match_batch_device_aux(adc_engine* e, int32_t n, const uint8_t* d_left, const uint8_t* d_right,
                               float* d_disp, const adc_aux_outputs* aux, void* stream);

/* Asynchronous host-buffer form for callers that pipeline their own I/O: buffers must be pinned
 * (adc_host_alloc or cudaHostAlloc / cudaHostRegister).  Enqueues H2D, compute and D2H, joined on
 * `stream`, without synchronising. */
int adc_match_batch_pinned_async(adc_engine* e, int32_t n, const uint8_t* left, const uint8_t* right,
                                 float* disp, void* stream);

/* Streaming use (SURVEY.md 8f rank 1): by default every async batch call makes `stream` wait for all of its work, so
 * two calls in a row drain the engine in between (the last waves of a call end in latency-bound refinement kernels with
 * nothing left to overlap them with).  In pipelined mode a batch call returns without that join: the next call's first
 * waves start on the lanes that are already free, and the caller makes its stream wait once, with adc_join, before it
 * touches any result.  Inputs are still consumed in stream order of the call; outputs of a call are complete only
 * after adc_join (or adc_synchronize).  Has no effect on the synchronous entry points. */
int adc_set_pipelined(adc_engine* e, int32_t on);
int adc_join(adc_engine* e, void* stream);

void* adc_host_alloc(size_t bytes);  /* pinned host memory (cudaHostAlloc) */
void  adc_host_free(void* p);
int   adc_synchronize(adc_engine* e);

/* number of kernel launches issued by this engine since creation (bench.py's gpu_launches) */
uint64_t adc_launch_count(const adc_engine* e);
/* per-stage device milliseconds of the most recent adc_match call (CUDA events):
 * out[0..5] = cost, aggregation, scanline, wta, refine, output copy -- the six figures the
 * reference prints from Match (ADCensusStereo.cpp:88-129). */
int adc_last_stage_ms(const adc_engine* e, float out[6]);
/* resolved configuration (wave_pairs, lanes, ...) */
int adc_get_config(const adc_engine* e, adc_config* out);

/* Times one kernel of the pipeline in isolation on the engine's own stream (CUDA events), over one
 * wave of wave_pairs pairs: kernel_id 0 = cost volume, 1 = horizontal arm sum, 2 = vertical arm sum
 * with division, 3 = scanline pass along x, 4 = scanline pass along y, 5 = WTA left+right, 6 / 7 = the fused
 * vertical / horizontal double pass of the aggregation (divide + sum, intermediate in shared memory), 8 = horizontal
 * arm sum with division, 9 = vertical arm sum without division, 10 = WTA left+right that also writes the side outputs
 * cost_best, cost_second and the WTA-invalid flag of the origin map.
 * algorithmic_bytes (optional) receives the bytes one launch must move (SURVEY.md section 8d). */
int adc_profile_kernel(adc_engine* e, int32_t kernel_id, int32_t reps, float* avg_ms, double* algorithmic_bytes);

/* Output side of the reference's demo program (main.cpp, outside ADCensusStereo itself; SURVEY.md 8f):
 *   adc_render_disparity = ShowDisparityMap / SaveDisparityMap (main.cpp:147-207): the 8-bit image
 *       uchar((|d| - min) / (max - min) * 255) with min / max over the valid pixels (0 where d is Invalid_Float),
 *       and that image through cv::COLORMAP_JET as packed BGR.  gray8 [W*H], jet_bgr [W*H*3], min_max [2]; any
 *       of the three may be NULL.  The file encoding (PNG) stays with the caller.
 *   adc_disparity_cloud = SaveDisparityCloud (main.cpp:209-230): one record (x, y, |d|, r, g, b) as six floats per
 *       valid pixel in raster order; `cloud` must hold W*H*6 floats, *n_points receives the record count.  The
 *       text formatting ("%f %f %f %d %d %d") stays with the caller.
 * Host pointers; the engine's lane 0 is used, so not concurrently with adc_match on the same engine. */
int adc_render_disparity(adc_engine* e, const float* disp, uint8_t* gray8, uint8_t* jet_bgr, float* min_max);
int adc_disparity_cloud(adc_engine* e, const uint8_t* img_left, const float* disp, float* cloud, int32_t* n_points);

const char* adc_last_error(void);
const char* adc_version(void);

/* ---- debug taps (parity tests) -------------------------------------------------------------
 * adc_debug_run executes the production pipeline on ONE pair up to and including `last_stage` and leaves every
 * buffer live (a run that stops between two aggregation iterations, AGG1..AGG3, takes the eight single aggregation
 * passes instead of the fused same-axis passes, whose intermediate never reaches memory); adc_debug_get copies a buffer out in the
 * reference's layout ([H][W][D] with d fastest for the volumes).  Stage and tap ids follow the
 * reference's structure: stages are the steps of Match / Aggregate / Optimize / Refine, taps are
 * the private members a parity test wants to see (cost_computor.h:80-91, cross_aggregator.h:88-102,
 * ADCensusStereo.h:88-92, multistep_refiner.h:96-99). */
enum {
    ADC_STAGE_COST = 0, ADC_STAGE_ARMS = 1,
    ADC_STAGE_AGG1 = 2, ADC_STAGE_AGG2 = 3, ADC_STAGE_AGG3 = 4, ADC_STAGE_AGG4 = 5,
    ADC_STAGE_SO1 = 6, ADC_STAGE_SO2 = 7, ADC_STAGE_SO3 = 8, ADC_STAGE_SO4 = 9,
    ADC_STAGE_WTA = 10, ADC_STAGE_OUTLIER = 11, ADC_STAGE_VOTE = 12, ADC_STAGE_INTERP = 13,
    ADC_STAGE_DISC = 14, ADC_STAGE_MEDIAN = 15, ADC_STAGE_COUNT = 16
};
enum {
    ADC_TAP_GRAY_L = 0, ADC_TAP_GRAY_R = 1,       /* u8  [H][W] */
    ADC_TAP_CENSUS_L = 2, ADC_TAP_CENSUS_R = 3,   /* u64 [H][W] */
    ADC_TAP_VOL_INIT = 4, ADC_TAP_VOL_AGGR = 5,   /* f32 [H][W][D]  (reference cost_init_ / cost_aggr_) */
    ADC_TAP_ARMS = 6,                             /* u8  [H][W][4]  left,right,top,bottom */
    ADC_TAP_SUPCNT_H = 7, ADC_TAP_SUPCNT_V = 8,   /* u16 [H][W] */
    ADC_TAP_DISP_L = 9, ADC_TAP_DISP_R = 10,      /* f32 [H][W] */
    ADC_TAP_MISMATCHES = 11, ADC_TAP_OCCLUSIONS = 12, /* i32 [n][2] (x,y), list order */
    ADC_TAP_COUNT = 13
};
int adc_debug_run(adc_engine* e, const uint8_t* img_left, const uint8_t* img_right, int32_t last_stage);
/* region-voting statistics of pair 0 of the last run: out[0],out[1] = remaining mismatch / occlusion
 * list sizes, out[2] = fixed-point rounds, out[3] = vote evaluations, out[12..15] = microseconds one warp spent
 * evaluating / waiting at round barriers / committing / compacting lists */
int adc_debug_counters(adc_engine* e, int32_t out[16]);
/* returns the tap's size in bytes (also when dst is NULL or cap is too small), 0 on error */
size_t adc_debug_get(adc_engine* e, int32_t tap, void* dst, size_t cap);

#ifdef __cplusplus
}
#endif
#endif /* ADCENSUS_B200_H_ */
