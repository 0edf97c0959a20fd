// adc_common.cuh -- shared declarations for the sm_100a AD-Census kernels.
//
// Data layout in HBM (per wave of S stereo pairs; every array is [S][...], pair index outermost):
//   bgr      u8  [S][2][H][W][3]   left, right packed BGR exactly as the caller passes them
//   gray     u8  [S][2][H][W]
//   census   u64 [S][2][H][W]
//   volA/B   f32 [S][H][W][Dp]     the two cost volumes, d fastest, Dp = D rounded up to 4 so that
//                                  every pixel's disparity vector is a whole number of 128-bit words
//   arms     u8x4[S][H][W]         left,right,top,bottom (cross_aggregator.h:17-20)
//   sup_h/v  u16 [S][H][W]
//   dmap     u8  [S][4][H][W]      colour-difference maps used by the scanline optimiser
//   disp_*   f32 [S][H][W]
//   label    u8  [S][H][W]         0 = valid, 1 = mismatch list, 2 = occlusion list
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define ADC_INVALID_F (__int_as_float(0x7f800000))  // +inf  (adcensus_types.h:33)
#define ADC_LARGE_F 99999.0f                         // adcensus_types.h:35
#define ADC_CNT 16                                   // ints of per-pair counters

struct AdcDims {
    int W, H, D, Dp;        // Dp: padded disparity stride (multiple of 4)
    int dmin, dmax;
    int N;                  // W*H
    long long vol_stride;   // floats per pair volume = N*Dp
};

// Everything a kernel may need from ADCensusOption plus derived constants, passed by value.
struct AdcParams {
    AdcDims dm;
    int L1, L2, t1, t2;          // cross arm parameters (L1 already clamped to 255)
    float p1, p2, p1_4, p2_4, p1_10, p2_10;  // so_p1/so_p2 and their /4, /10 quotients (IEEE, host-computed)
    int tso;
    int irv_ts; float irv_th;
    float lr_thres;
    int max_search;              // max(|dmax|,|dmin|)
    int dbg;                     // adc_config.debug_flags (test hooks, ADC_DBG_* in adcensus_b200.h)
};

__device__ __forceinline__ int adc_colour_dist(uchar3 a, uchar3 b) {
    int d0 = abs((int)a.x - (int)b.x), d1 = abs((int)a.y - (int)b.y), d2 = abs((int)a.z - (int)b.z);
    return max(d0, max(d1, d2));
}

__device__ __forceinline__ uchar3 adc_load_bgr(const uint8_t* __restrict__ img, int idx) {
    const uint8_t* p = img + 3ll * idx;
    return make_uchar3(__ldg(p), __ldg(p + 1), __ldg(p + 2));
}

// order-preserving float -> uint key (any sign), for REDUX-based warp minima
__device__ __forceinline__ unsigned adc_f2key(float f) {
    unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float adc_key2f(unsigned k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// Function attributes and __device__ / __constant__ symbols exist once per device: one-time set-up is keyed by the
// current device (one process may own engines on several GPUs, driven from several threads: the flags are atomics, and
// a thread that loses the race may run the kernel before the winner's attribute call has returned -- so every caller
// that finds the flag unset performs the (idempotent) set-up itself, and the flag is only published afterwards).
#include <atomic>
struct AdcOnce { std::atomic<int> done[64]; };
inline bool adc_once_needed(AdcOnce& o) {
    int dev = 0;
    cudaGetDevice(&dev);
    return o.done[dev & 63].load(std::memory_order_acquire) == 0;
}
inline void adc_once_done(AdcOnce& o) {
    int dev = 0;
    cudaGetDevice(&dev);
    o.done[dev & 63].store(1, std::memory_order_release);
}

// TMA descriptors (CUtensorMap, 128 bytes each) of a lane's two cost volumes for the two axes of the fused aggregation kernel
struct alignas(64) AdcArmTmaps { unsigned char map[2][2][128]; int ok; };

// ---- launchers (defined in the k_*.cu files; all asynchronous on `st`) -------------------------
struct AdcWave {            // device pointers of one wave (S pairs)
    int S;                  // active pairs in this launch
    uint8_t* bgr;           // [S][2][N*3]
    unsigned* bgrx;         // [S][2][N] the same pixels packed B | G<<8 | R<<16 (one 32-bit load per pixel)
    uint8_t* gray;          // [S][2][N]
    unsigned long long* census; // [S][2][N]
    float* volA; float* volB;
    uchar4* arms;
    const AdcArmTmaps* arm_tm;   // host memory, owned by the lane (NULL: the fused kernel loads its source with LDG)
    unsigned* arm_rec;      // [S][window records of both axes] which of a group's four outputs takes which tap (k_aggregate.cu)
    uint16_t* sup_h; uint16_t* sup_v;
    uint8_t* dmap;          // [S][4][N]: 0 = left-horizontal, 1 = left-vertical, 2 = right-horizontal, 3 = right-vertical
    float* disp_l; float* disp_r; float* disp_t;
    uint8_t* label; uint8_t* flag;
    int* pend;              // [S][2][N] mismatch / occlusion pixel lists (raster order)
    int* vlist;             // [S][2][N] the sub-lists region voting works on (pixels that can still be filled)
    int* counters;          // [S][ADC_CNT]: 0,1 list sizes; 2 voting rounds; 3 voting evaluations; 4.. flags/queues
    int* rowcnt;            // [S][2][H] per-row list counts / offsets
    unsigned* so_bitrows;   // [S][4][H][row words] mirrored per-row bit vectors of the right image (scanline optimiser)
    unsigned* so_rec;       // [S][4][N][rec words] per-pixel penalty records of the four pass directions
    int* tile_stamp;        // [S][tiles] region voting: epoch of the last change near a 16x16 tile
    int* last_eval;         // [S][N]     region voting: epoch of a pixel's (or tile's) last evaluation
    unsigned long long* wta_key;  // [S][N] right-view WTA keys (ordered cost << 32 | disparity index)
    int2* vote_dirty;       // [S][N]     region voting: work list of the current round
    uchar2* vote_alr;       // [S][N]     region voting: horizontal arms only (left, right)
    uint8_t* vote_dq;       // [S][2][N]  region voting: rounded disparity index per pixel, NEW and OLD state
    uchar2* vote_atbT;      // [S][W][H]  region voting: vertical arms (top, bottom), transposed (a column is contiguous)
    int* vote_pslotT;       // [S][W][H]  region voting: histogram slot of a pending pixel, -1 otherwise (transposed)
    uint8_t* vote_val;      // [S][N]     region voting: current vote per slot (255 = none)
    uint8_t* vote_dirtyb;   // [S][N]     region voting: slot's histogram changed since its last derive
    int* vote_state;        // [S][N]     region voting: disparity index of a valid pixel, -1 invalid, -(slot+2) pending
    int* vote_deg;          // [S][N]     region voting: adjacency list lengths / fill cursors per slot
    int* vote_off;          // [S][N+1]   region voting: adjacency list offsets (CSR by target slot)
    unsigned* vote_hist;    // [S][vol_stride] region voting: histograms + forward lists + adjacency (= volB, idle after the last scanline pass)
    const float* lut_ad;    // [766]  (1 - exp(-(s/3)/lambda_ad)) + 1, host libm expf
    const float* lut_cen;   // [64]   exp(-h/lambda_census)
    const double* ray_sin; const double* ray_cos; // [16] host libm sin/cos of the accumulated angles
    const short2* ray_off;  // [16][max_search] (dx,dy) = (lround(m*cos), lround(m*sin)); NULL if not verified exact
};

void adc_launch_gray_census(const AdcParams& P, const AdcWave& w, cudaStream_t st, unsigned long long* launches);
void adc_launch_cost(const AdcParams& P, const AdcWave& w, float* vol, cudaStream_t st, unsigned long long* launches);
void adc_launch_diffmaps(const AdcParams& P, const AdcWave& w, cudaStream_t st, unsigned long long* launches);
void adc_launch_arms(const AdcParams& P, const AdcWave& w, cudaStream_t st, unsigned long long* launches);
// one 1-D pass of the cross aggregation: horizontal (dir=0) or vertical (dir=1) ordered sums,
// optionally divided by the support count `sup` (second pass of an iteration)
void adc_launch_arm_sum(const AdcParams& P, const AdcWave& w, const float* src, float* dst, int dir,
                        const uint16_t* sup, cudaStream_t st, unsigned long long* launches);
// two consecutive passes along the same axis (second pass of an iteration, divided by `sup_mid`, then the first pass of the
// next iteration) with the intermediate kept in shared memory; false = not applicable for these parameters, nothing launched
bool adc_arm_sum2_available(const AdcParams& P);
bool adc_launch_arm_sum2(const AdcParams& P, const AdcWave& w, const float* src, float* dst, int dir,
                         const uint16_t* sup_mid, cudaStream_t st, unsigned long long* launches);
size_t adc_arm_rec_bytes(const AdcDims& dm, int L1);   // window records of one pair
bool adc_arm_tmaps_encode(const AdcParams& P, int S, float* volA, float* volB, AdcArmTmaps* out);   // false: TMA path not available
size_t adc_arm_overread_floats(const AdcDims& dm);     // padding the arena keeps behind the two volumes
void adc_launch_so_bitrows(const AdcParams& P, const AdcWave& w, cudaStream_t st, unsigned long long* launches);
size_t adc_so_rec_bytes(const AdcDims& dm);
size_t adc_so_bitrow_bytes(const AdcDims& dm);
// one scanline pass: (sx,sy) in {(1,0),(-1,0),(0,1),(0,-1)}
int adc_launch_scanline(const AdcParams& P, const AdcWave& w, const float* src, float* dst, int sx, int sy,
                        cudaStream_t st, unsigned long long* launches);
int adc_launch_wta(const AdcParams& P, const AdcWave& w, const float* vol, cudaStream_t st, unsigned long long* launches);
// Device buffers of the side outputs of one wave ([S][N] each; NULL = not wanted).  `origin` is written in two steps: the
// WTA kernel stores the WTA-invalid flag, adc_launch_origin ORs the code on; `lab0` keeps the outlier labels from
// before region voting (only with `origin`).
struct AdcAux {
    uint8_t* origin;
    uint8_t* lab0;
    float* cost_best;
    float* cost_second;
};
// the same WTA, also writing cost_best / cost_second / the WTA-invalid flag of the left view where aux asks for them
int adc_launch_wta_aux(const AdcParams& P, const AdcWave& w, const float* vol, const AdcAux& aux, cudaStream_t st,
                       unsigned long long* launches);
// origin code of every pixel from aux.lab0, the labels after voting (w.label) and the map after the last filling step
// (w.disp_l)
void adc_launch_origin(const AdcParams& P, const AdcWave& w, const AdcAux& aux, cudaStream_t st, unsigned long long* launches);
void adc_launch_outlier(const AdcParams& P, const AdcWave& w, cudaStream_t st, unsigned long long* launches);
void adc_launch_build_lists(const AdcParams& P, const AdcWave& w, cudaStream_t st, unsigned long long* launches);
void adc_launch_voting(const AdcParams& P, const AdcWave& w, cudaStream_t st, unsigned long long* launches);
// incremental-histogram voting (k_vote.cu); expects the active lists (w.vlist, counters 10/11) and the byte state
// (w.vote_dq, w.vote_alr); uses w.volB as histogram storage.  false = not applicable, nothing launched
bool adc_launch_vote_push(const AdcParams& P, const AdcWave& w, cudaStream_t st, unsigned long long* launches);
// k = 0: mismatch list, k = 1: occlusion list; reads disp_l, writes disp_t
void adc_launch_interp_list(const AdcParams& P, const AdcWave& w, int k, cudaStream_t st, unsigned long long* launches);
void adc_launch_discontinuity(const AdcParams& P, const AdcWave& w, const float* vol, cudaStream_t st, unsigned long long* launches);
// in-place-equivalent 3x3 median: reads `in`, writes `out` (different buffers); non-zero if H is too large
// output side of the demo (k_render.cu): 8-bit normalised map + JET colouring; (x,y,d,r,g,b) cloud of the valid pixels
int adc_launch_render(const AdcDims& dm, const float* d_disp, unsigned* d_mm, uint8_t* d_gray, uint8_t* d_jet, float* d_mm_out,
                      cudaStream_t st, unsigned long long* launches);
void adc_launch_cloud(const AdcParams& P, const AdcWave& w1, const float* d_disp, const uint8_t* d_bgr, float* d_cloud,
                      cudaStream_t st, unsigned long long* launches);
int adc_launch_median(const AdcParams& P, const AdcWave& w, const float* in, float* out, cudaStream_t st,
                      unsigned long long* launches);
// Dynamic shared memory one launch of the kernel needs at these sizes, and in *cap the most its function attribute
// grants (adc_create refuses sizes for which need > cap)
size_t adc_cost_smem(const AdcDims& dm, size_t* cap);
size_t adc_scanline_smem(const AdcDims& dm, size_t* cap);
size_t adc_voting_smem(const AdcDims& dm, size_t* cap);
