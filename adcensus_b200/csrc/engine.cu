// engine.cu -- host side of the B200 AD-Census engine and its C ABI (include/adcensus_b200.h).
//
// An engine owns `lanes` independent pipelines.  A lane = one CUDA stream + a device arena for a
// wave of up to `wave_pairs` stereo pairs (two cost volumes per pair dominate: 2*4*N*Dp bytes) +
// pinned staging for callers that hand in pageable memory.  A batch is cut into waves that are
// dealt round-robin to the lanes; every kernel of a wave is one batched launch over all its pairs
// (pair index = outermost grid dimension), and the lanes overlap each other's copies, bandwidth
// kernels and the latency-bound refinement kernels.  Nothing here ever falls back to a CPU path:
// if the CUDA library cannot run, the call fails.
#include <cuda_runtime.h>

#include <math.h>
#include <stdarg.h>
#include <stddef.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/adcensus_b200.h"
#include "adc_common.cuh"

static_assert(sizeof(adc_option) == 60, "adc_option must match the reference's ADCensusOption (60 bytes)");
static_assert(offsetof(adc_option, so_p1) == 32 && offsetof(adc_option, irv_th) == 48 &&
              offsetof(adc_option, do_lr_check) == 56 && offsetof(adc_option, do_discontinuity_adjustment) == 58,
              "adc_option field offsets must match adcensus_types.h:45-75");
static_assert(sizeof(adc_config) == 64 && offsetof(adc_config, max_disparity_range) == 16,
              "adc_config layout is part of the ABI: 64 bytes, max_disparity_range at offset 16");
static_assert(sizeof(adc_aux_outputs) == 32 && offsetof(adc_aux_outputs, origin) == 0 &&
              offsetof(adc_aux_outputs, cost_best) == 8 && offsetof(adc_aux_outputs, cost_second) == 16 &&
              offsetof(adc_aux_outputs, disp_right) == 24, "adc_aux_outputs layout is part of the ABI: four pointers, 32 bytes");

namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CK(call)                                                                                 \
    do {                                                                                         \
        cudaError_t err__ = (call);                                                              \
        if (err__ != cudaSuccess)                                                                \
            return fail(ADC_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(err__), __FILE__, __LINE__); \
    } while (0)

struct Lane {
    cudaStream_t st = nullptr;
    cudaEvent_t ev_done = nullptr;     // all work of the lane's latest wave (incl. D2H) finished
    cudaEvent_t ev_in_free = nullptr;  // the H2D of the latest wave has consumed the staging-in buffer
    void* arena = nullptr;
    AdcWave w{};                       // device pointers, capacity S pairs
    AdcArmTmaps arm_tm{};              // TMA descriptors of this lane's volumes (fused aggregation kernel)
    uint8_t* pin_in = nullptr;         // [S][2][N*3] pinned staging (pageable callers only)
    float* pin_out = nullptr;          // [S][N]
    // pending copy-out of a staged wave (pageable callers)
    int drain_n = 0;
    float* const* drain_ptrs = nullptr;
    float* drain_base = nullptr;
    int drain_first = 0;
    // side outputs, allocated by the first call that asks for them (ensure_aux)
    void* aux_arena = nullptr;         // device scratch of the wave: origin, lab0, cost_best, cost_second, [S][N] each
    AdcAux aux{};
    void* aux_pin = nullptr;           // pinned staging of the four outputs (pageable callers)
    adc_aux_outputs pin_aux{};         // ... carved: origin, cost_best, cost_second, disp_right, [S][N] each
    adc_aux_outputs drain_aux{};       // the caller's side-output buffers of the pending copy-out (NULL members: none)
};

}  // namespace

struct adc_engine {
    int W = 0, H = 0;
    adc_option opt{};
    adc_config cfg{};
    AdcParams P{};
    int S = 0;
    std::vector<Lane> lanes;
    cudaStream_t main_st = nullptr;
    cudaEvent_t ev_fork = nullptr;
    float* d_lut_ad = nullptr;
    float* d_lut_cen = nullptr;
    double* d_rays = nullptr;  // [32]: sin[16], cos[16]
    short2* d_ray_off = nullptr;  // [16][max_search] integer ray offsets, when verified exact for this image size
    bool pipelined = false;            // adc_set_pipelined: batch calls do not join the caller's stream themselves
    bool agg_fused = false;            // same-axis aggregation passes of neighbouring iterations run as one kernel (k_arm_sum2)
    unsigned long long launches = 0;
    float stage_ms[6] = {0, 0, 0, 0, 0, 0};
    cudaEvent_t ev_stage[8] = {};
    // debug state (adc_debug_run): which buffer plays the reference's cost_init_ / cost_aggr_
    const float* dbg_init = nullptr;
    const float* dbg_aggr = nullptr;
    int dbg_stage = -1;
};

namespace {

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct Carver {
    char* base;
    size_t off = 0;
    explicit Carver(void* b) : base(static_cast<char*>(b)) {}
    template <typename T> T* take(size_t count) {
        T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
        off = align_up(off + count * sizeof(T), 256);
        return p;
    }
};

// Carves (or, with base == nullptr, just sizes) one lane's arena.
size_t carve_lane(void* base, const AdcDims& dm, int L1, int S, AdcWave* w) {
    Carver c(base);
    const size_t N = (size_t)dm.N;
    AdcWave t{};
    t.volA = c.take<float>((size_t)S * dm.vol_stride);
    t.volB = c.take<float>((size_t)S * dm.vol_stride);
    c.take<float>(adc_arm_overread_floats(dm));           // the arm-sum walks may load (never use) a few taps past a volume's end
    t.bgr = c.take<uint8_t>((size_t)S * 2 * N * 3);
    t.gray = c.take<uint8_t>((size_t)S * 2 * N);
    t.bgrx = c.take<unsigned>((size_t)S * 2 * N);
    t.census = c.take<unsigned long long>((size_t)S * 2 * N);
    t.arms = c.take<uchar4>((size_t)S * N);
    t.arm_rec = c.take<unsigned>((size_t)S * adc_arm_rec_bytes(dm, L1) / 4);
    t.sup_h = c.take<uint16_t>((size_t)S * N);
    t.sup_v = c.take<uint16_t>((size_t)S * N);
    t.dmap = c.take<uint8_t>((size_t)S * 4 * N);
    t.disp_l = c.take<float>((size_t)S * N);
    t.disp_r = c.take<float>((size_t)S * N);
    t.disp_t = c.take<float>((size_t)S * N);
    t.label = c.take<uint8_t>((size_t)S * N);
    t.flag = c.take<uint8_t>((size_t)S * N);
    t.pend = c.take<int>((size_t)S * 2 * N);
    t.vlist = c.take<int>((size_t)S * 2 * N);
    t.counters = c.take<int>((size_t)S * ADC_CNT);
    t.vote_dq = c.take<uint8_t>((size_t)S * 2 * N);
    t.vote_alr = c.take<uchar2>((size_t)S * N);
    t.vote_dirty = c.take<int2>((size_t)S * N);
    t.vote_atbT = c.take<uchar2>((size_t)S * N);
    t.vote_pslotT = c.take<int>((size_t)S * N);
    t.vote_val = c.take<uint8_t>((size_t)S * N);
    t.vote_dirtyb = c.take<uint8_t>((size_t)S * N);
    t.vote_state = c.take<int>((size_t)S * N);
    t.vote_deg = c.take<int>((size_t)S * N);
    t.vote_off = c.take<int>((size_t)S * (N + 1));
    t.wta_key = c.take<unsigned long long>((size_t)S * N);
    t.rowcnt = c.take<int>((size_t)S * 2 * dm.H);
    t.so_bitrows = c.take<unsigned>((size_t)S * adc_so_bitrow_bytes(dm) / 4);
    t.so_rec = c.take<unsigned>((size_t)S * adc_so_rec_bytes(dm) / 4);
    t.tile_stamp = c.take<int>((size_t)S * ((dm.W + 15) / 16) * ((dm.H + 15) / 16));
    t.last_eval = c.take<int>((size_t)S * N);
    t.vote_hist = reinterpret_cast<unsigned*>(t.volB);   // idle after the last scanline pass
    if (w) *w = t;
    return c.off;
}

void build_params(adc_engine* e) {
    const adc_option& o = e->opt;
    AdcParams& P = e->P;
    P.dm.W = e->W; P.dm.H = e->H;
    P.dm.dmin = o.min_disparity; P.dm.dmax = o.max_disparity;
    P.dm.D = o.max_disparity - o.min_disparity;
    P.dm.Dp = (P.dm.D + 3) / 4 * 4;
    P.dm.N = e->W * e->H;
    P.dm.vol_stride = (long long)P.dm.N * P.dm.Dp;
    P.L1 = std::min(o.cross_L1, 255);  // min(cross_L1_, MAX_ARM_LENGTH), cross_aggregator.cpp:151
    P.L2 = o.cross_L2; P.t1 = o.cross_t1; P.t2 = o.cross_t2;
    // scanline_optimizer.cpp:133-140: p/4 and p/10 are float / int -> IEEE float division
    P.p1 = o.so_p1; P.p2 = o.so_p2;
    P.p1_4 = o.so_p1 / 4; P.p2_4 = o.so_p2 / 4;
    P.p1_10 = o.so_p1 / 10; P.p2_10 = o.so_p2 / 10;
    P.tso = o.so_tso;
    P.irv_ts = o.irv_ts; P.irv_th = o.irv_th;
    P.lr_thres = o.lrcheck_thres;
    P.max_search = std::max(abs(o.max_disparity), abs(o.min_disparity));  // multistep_refiner.cpp:236
    P.dbg = e->cfg.debug_flags;
}

int upload_tables(adc_engine* e) {
    // exp() factors of the AD-census cost on their integer domains, with THIS host's libm expf and
    // the reference's operation order (cost_computor.cpp:110-117): the device never calls exp.
    std::vector<float> ad(766), cen(64);
    for (int s = 0; s < 766; s++) {
        const float cost_ad = (float)s / 3.0f;
        const float e_ad = expf(-cost_ad / (float)e->opt.lambda_ad);
        float t = 1.0f - e_ad;
        t = t + 1.0f;
        ad[s] = t;
    }
    for (int h = 0; h < 64; h++) cen[h] = expf(-(float)h / (float)e->opt.lambda_census);
    // ray directions of ProperInterpolation (multistep_refiner.cpp:234,252-254,268)
    double rays[32];
    const float pi = 3.1415926f;
    double ang = 0.0;
    for (int s = 0; s < 16; s++) {
        rays[s] = sin(ang);
        rays[16 + s] = cos(ang);
        ang += pi / 16;
    }
    CK(cudaMalloc(&e->d_lut_ad, sizeof(float) * 766));
    CK(cudaMalloc(&e->d_lut_cen, sizeof(float) * 64));
    CK(cudaMalloc(&e->d_rays, sizeof(double) * 32));
    CK(cudaMemcpy(e->d_lut_ad, ad.data(), sizeof(float) * 766, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(e->d_lut_cen, cen.data(), sizeof(float) * 64, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(e->d_rays, rays, sizeof(double) * 32, cudaMemcpyHostToDevice));
    // ProperInterpolation evaluates lround(y + m*sin) per step (multistep_refiner.cpp:252-254).  For integer y
    // that equals y + lround(m*sin) unless a rounding of the double sum (or a half-way case) intervenes;
    // check every (ray, m, coordinate) the image can produce and only then let the kernel use the table.
    const int L = e->P.max_search;
    if (L > 1 && L < 4096 && !(e->cfg.debug_flags & ADC_DBG_NO_RAY_TABLE)) {
        std::vector<short2> off((size_t)16 * L);
        bool exact = true;
        for (int s = 0; s < 16 && exact; s++)
            for (int m = 1; m < L && exact; m++) {
                const long dy = lround(m * rays[s]), dx = lround(m * rays[16 + s]);
                for (int y = 0; y < e->H && exact; y++) exact = lround(y + m * rays[s]) == y + dy;
                for (int x = 0; x < e->W && exact; x++) exact = lround(x + m * rays[16 + s]) == x + dx;
                off[(size_t)s * L + m] = make_short2((short)dx, (short)dy);
            }
        if (exact) {
            CK(cudaMalloc(&e->d_ray_off, sizeof(short2) * off.size()));
            CK(cudaMemcpy(e->d_ray_off, off.data(), sizeof(short2) * off.size(), cudaMemcpyHostToDevice));
        }
    }
    return ADC_OK;
}

AdcWave wave_view(const adc_engine* e, const Lane& ln, int nS) {
    AdcWave w = ln.w;
    w.S = nS;
    w.lut_ad = e->d_lut_ad;
    w.lut_cen = e->d_lut_cen;
    w.ray_sin = e->d_rays;
    w.ray_cos = e->d_rays + 16;
    w.ray_off = e->d_ray_off;
    return w;
}

// Enqueues the whole pipeline for the nS pairs whose images already sit in ln.w.bgr.  Stops after
// `last_stage` (ADC_STAGE_MEDIAN = everything).  ev[] (optional, 6 events) are recorded at the
// stage boundaries the reference times in Match (ADCensusStereo.cpp:81-129).
// `aux` (optional): device buffers of the side outputs this run writes besides the map; NULL = the plain pipeline.
int enqueue_pipeline(adc_engine* e, Lane& ln, int nS, int last_stage, cudaEvent_t* ev, const AdcAux* aux = nullptr) {
    const AdcParams& P = e->P;
    const AdcWave w = wave_view(e, ln, nS);
    cudaStream_t st = ln.st;
    unsigned long long* L = &e->launches;
    const size_t mapN = (size_t)nS * P.dm.N;
    // The two volumes play the reference's cost_init_ / cost_aggr_.  The aggregation leaves its result in volA either way:
    //   eight single passes:   cost -> A | H: A->B, V/: B->A | V: A->B, H/: B->A | ...                          (8 x 2 = 16 volume transfers)
    //   same-axis passes fused (second pass of iteration k + first pass of iteration k+1 in one kernel):
    //                          cost -> B | H: B->A | V/ V: A->B | H/ H: B->A | V/ V: A->B | H/: B->A           (5 x 2 = 10 volume transfers)
    // A run that has to stop between iterations (debug taps AGG1..AGG3) takes the single passes.
    const bool fused = e->agg_fused && !(last_stage >= ADC_STAGE_AGG1 && last_stage <= ADC_STAGE_AGG3);
    float* A = w.volA;
    float* B = w.volB;
    float* C0 = fused ? B : A;          // where the cost volume is written
    e->dbg_init = C0;
    e->dbg_aggr = C0;
    auto stop = [&](int stage) { e->dbg_stage = stage; return stage >= last_stage; };
    // launch errors surface where they happen: a stage boundary reports the first failed launch since the previous one
    auto launched = [&](const char* what) -> int {
        const cudaError_t err = cudaGetLastError();
        if (err != cudaSuccess) return fail(ADC_ERR_CUDA, "%s: kernel launch failed: %s", what, cudaGetErrorString(err));
        return ADC_OK;
    };
    int rc;

    // ---- stage 1: cost (cost_computor.cpp:123-137)
    adc_launch_gray_census(P, w, st, L);
    adc_launch_cost(P, w, C0, st, L);
    if ((rc = launched("cost volume"))) return rc;
    if (ev) CK(cudaEventRecord(ev[1], st));
    if (stop(ADC_STAGE_COST)) return ADC_OK;

    // ---- stage 2: arms, support counts, window records, 4 aggregation iterations (cross_aggregator.cpp:89-118)
    adc_launch_arms(P, w, st, L);
    if ((rc = launched("cross arms"))) return rc;
    if (stop(ADC_STAGE_ARMS)) return ADC_OK;
    if (fused) {
        adc_launch_arm_sum(P, w, B, A, 0, nullptr, st, L);                       // it 0: H
        if (!adc_launch_arm_sum2(P, w, A, B, 1, w.sup_h, st, L) ||               // it 0: V /   + it 1: V
            !adc_launch_arm_sum2(P, w, B, A, 0, w.sup_v, st, L) ||               // it 1: H /   + it 2: H
            !adc_launch_arm_sum2(P, w, A, B, 1, w.sup_h, st, L))                 // it 2: V /   + it 3: V
            return fail(ADC_ERR_UNSUPPORTED, "fused aggregation pass not applicable");
        adc_launch_arm_sum(P, w, B, A, 0, w.sup_v, st, L);                       // it 3: H /
        e->dbg_aggr = A;
        e->dbg_stage = ADC_STAGE_AGG4;
    } else {
        for (int it = 0; it < 4; it++) {
            const bool hfirst = (it % 2) == 0;  // H,V | V,H | H,V | V,H  (:102,116)
            adc_launch_arm_sum(P, w, A, B, hfirst ? 0 : 1, nullptr, st, L);
            adc_launch_arm_sum(P, w, B, A, hfirst ? 1 : 0, hfirst ? w.sup_h : w.sup_v, st, L);
            if (stop(ADC_STAGE_AGG1 + it)) return launched("aggregation");
        }
    }
    if ((rc = launched("aggregation"))) return rc;
    if (ev) CK(cudaEventRecord(ev[2], st));
    if (last_stage <= ADC_STAGE_AGG4) return ADC_OK;

    // ---- stage 3: scanline optimisation, 4 chained passes (scanline_optimizer.cpp:54-60)
    adc_launch_diffmaps(P, w, st, L);
    adc_launch_so_bitrows(P, w, st, L);
    static const int dirs[4][2] = {{1, 0}, {-1, 0}, {0, 1}, {0, -1}};
    for (int ps = 0; ps < 4; ps++) {
        const float* src = (ps % 2 == 0) ? A : B;
        float* dst = (ps % 2 == 0) ? B : A;
        if (adc_launch_scanline(P, w, src, dst, dirs[ps][0], dirs[ps][1], st, L))
            return fail(ADC_ERR_UNSUPPORTED, "disparity range %d exceeds the scanline kernel's limit of %d", P.dm.D,
                        ADC_MAX_DISPARITY_RANGE_WIDE);
        if (ps % 2 == 0) e->dbg_init = B; else e->dbg_aggr = A;
        if (stop(ADC_STAGE_SO1 + ps)) return launched("scanline optimisation");
    }
    if ((rc = launched("scanline optimisation"))) return rc;
    if (ev) CK(cudaEventRecord(ev[3], st));

    // ---- stage 4: left + right disparity (ADCensusStereo.cpp:108-109)
    const bool wta_aux = aux && (aux->origin || aux->cost_best || aux->cost_second);
    if (wta_aux ? adc_launch_wta_aux(P, w, A, *aux, st, L) : adc_launch_wta(P, w, A, st, L))
        return fail(ADC_ERR_UNSUPPORTED, "WTA launch failed");
    if ((rc = launched("winner-takes-all"))) return rc;
    if (ev) CK(cudaEventRecord(ev[4], st));
    if (stop(ADC_STAGE_WTA)) return ADC_OK;

    // ---- stage 5: multi-step refinement (multistep_refiner.cpp:60-87)
    if (e->opt.do_lr_check) {
        adc_launch_outlier(P, w, st, L);  // disp_l (orig) -> disp_t, label
        CK(cudaMemcpyAsync(w.disp_l, w.disp_t, mapN * sizeof(float), cudaMemcpyDeviceToDevice, st));
    } else {
        CK(cudaMemsetAsync(w.label, 0, mapN, st));
        CK(cudaMemcpyAsync(w.disp_t, w.disp_l, mapN * sizeof(float), cudaMemcpyDeviceToDevice, st));
    }
    if (aux && aux->origin) CK(cudaMemcpyAsync(aux->lab0, w.label, mapN, cudaMemcpyDeviceToDevice, st));   // voting clears labels
    if (stop(ADC_STAGE_OUTLIER)) return launched("outlier detection");
    if (e->opt.do_filling) {  // gates voting AND interpolation (ADCensusStereo.cpp:183)
        CK(cudaMemsetAsync(w.counters, 0, (size_t)nS * ADC_CNT * sizeof(int), st));
        adc_launch_build_lists(P, w, st, L);
        adc_launch_voting(P, w, st, L);
        if ((rc = launched("region voting"))) return rc;
        if (stop(ADC_STAGE_VOTE)) return ADC_OK;
        for (int k = 0; k < 2; k++) {
            adc_launch_interp_list(P, w, k, st, L);
            CK(cudaMemcpyAsync(w.disp_l, w.disp_t, mapN * sizeof(float), cudaMemcpyDeviceToDevice, st));
        }
        if (stop(ADC_STAGE_INTERP)) return launched("interpolation");
    } else if (last_stage <= ADC_STAGE_INTERP) {
        e->dbg_stage = last_stage;
        return launched("refinement");
    }
    if (aux && aux->origin) adc_launch_origin(P, w, *aux, st, L);
    if (e->opt.do_discontinuity_adjustment) adc_launch_discontinuity(P, w, A, st, L);
    if (stop(ADC_STAGE_DISC)) return launched("discontinuity adjustment");
    // median: disp_l -> disp_t, then back so that disp_l always holds the current map
    if (adc_launch_median(P, w, w.disp_l, w.disp_t, st, L))
        return fail(ADC_ERR_UNSUPPORTED, "image height %d exceeds the median kernel's limit", P.dm.H);
    CK(cudaMemcpyAsync(w.disp_l, w.disp_t, mapN * sizeof(float), cudaMemcpyDeviceToDevice, st));
    if (ev) CK(cudaEventRecord(ev[5], st));
    e->dbg_stage = ADC_STAGE_MEDIAN;
    return launched("refinement");
}

bool is_pinned(const void* p) {
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost || at.type == cudaMemoryTypeManaged;
}

// ---- side outputs ----
bool aux_wanted(const adc_aux_outputs* a) { return a && (a->origin || a->cost_best || a->cost_second || a->disp_right); }
bool aux_needs_scratch(const adc_aux_outputs* a) { return a->origin || a->cost_best || a->cost_second; }

// The four outputs of an adc_aux_outputs as (buffer, bytes per pixel), in declaration order.
struct AuxOut { char* p; size_t el; };
void aux_outs(const adc_aux_outputs& a, AuxOut o[4]) {
    o[0] = {reinterpret_cast<char*>(a.origin), 1};
    o[1] = {reinterpret_cast<char*>(a.cost_best), 4};
    o[2] = {reinterpret_cast<char*>(a.cost_second), 4};
    o[3] = {reinterpret_cast<char*>(a.disp_right), 4};
}

// Device scratch of every lane (when the request needs more than disp_right) and pinned staging of the first
// `staging_lanes` lanes, allocated once, on the first call that needs them.  A failed allocation leaves the engine as it
// was, apart from what was already allocated (kept for the next call, freed by adc_destroy).
int ensure_aux(adc_engine* e, bool scratch, int staging_lanes) {
    const size_t SN = (size_t)e->S * e->P.dm.N;
    for (size_t li = 0; li < e->lanes.size(); li++) {
        Lane& ln = e->lanes[li];
        if (scratch && !ln.aux_arena) {
            Carver sz(nullptr);
            sz.take<uint8_t>(SN); sz.take<uint8_t>(SN); sz.take<float>(SN); sz.take<float>(SN);
            void* p = nullptr;
            if (cudaMalloc(&p, sz.off) != cudaSuccess) {
                cudaGetLastError();
                return fail(ADC_ERR_NOMEM, "side-output scratch of %zu bytes", sz.off);
            }
            Carver c(p);
            ln.aux.origin = c.take<uint8_t>(SN);
            ln.aux.lab0 = c.take<uint8_t>(SN);
            ln.aux.cost_best = c.take<float>(SN);
            ln.aux.cost_second = c.take<float>(SN);
            ln.aux_arena = p;
        }
        if ((int)li < staging_lanes && !ln.aux_pin) {
            Carver sz(nullptr);
            sz.take<uint8_t>(SN); sz.take<float>(SN); sz.take<float>(SN); sz.take<float>(SN);
            void* p = nullptr;
            if (cudaHostAlloc(&p, sz.off, cudaHostAllocDefault) != cudaSuccess) {
                cudaGetLastError();
                return fail(ADC_ERR_NOMEM, "pinned side-output staging of %zu bytes", sz.off);
            }
            Carver c(p);
            ln.pin_aux.origin = c.take<uint8_t>(SN);
            ln.pin_aux.cost_best = c.take<float>(SN);
            ln.pin_aux.cost_second = c.take<float>(SN);
            ln.pin_aux.disp_right = c.take<float>(SN);
            ln.aux_pin = p;
        }
    }
    return ADC_OK;
}

// The lane's device buffers for what `a` asks for (NULL members where it asks for nothing).
AdcAux wave_aux(const Lane& ln, const adc_aux_outputs& a) {
    AdcAux x{};
    if (a.origin) { x.origin = ln.aux.origin; x.lab0 = ln.aux.lab0; }
    if (a.cost_best) x.cost_best = ln.aux.cost_best;
    if (a.cost_second) x.cost_second = ln.aux.cost_second;
    return x;
}

// Enqueues the copies of the side outputs of nS pairs from the lane's wave into dst (pair `first` of the caller's arrays).
int copy_aux_out(const Lane& ln, const AdcAux& x, const adc_aux_outputs& dst, size_t first, int nS, size_t N,
                 cudaMemcpyKind kind, cudaStream_t st) {
    const void* src[4] = {x.origin, x.cost_best, x.cost_second, ln.w.disp_r};
    AuxOut o[4];
    aux_outs(dst, o);
    for (int k = 0; k < 4; k++)
        if (o[k].p) CK(cudaMemcpyAsync(o[k].p + first * N * o[k].el, src[k], (size_t)nS * N * o[k].el, kind, st));
    return ADC_OK;
}

// The lane's pinned staging for the members `want` asks for (NULL members elsewhere).
adc_aux_outputs staging_for(const Lane& ln, const adc_aux_outputs& want) {
    adc_aux_outputs s{};
    if (want.origin) s.origin = ln.pin_aux.origin;
    if (want.cost_best) s.cost_best = ln.pin_aux.cost_best;
    if (want.cost_second) s.cost_second = ln.pin_aux.cost_second;
    if (want.disp_right) s.disp_right = ln.pin_aux.disp_right;
    return s;
}

int drain_lane(adc_engine* e, Lane& ln) {
    if (ln.drain_n == 0) return ADC_OK;
    CK(cudaEventSynchronize(ln.ev_done));
    const size_t N = (size_t)e->P.dm.N;
    for (int i = 0; i < ln.drain_n; i++) {
        float* dst = ln.drain_ptrs ? ln.drain_ptrs[ln.drain_first + i] : ln.drain_base + (size_t)(ln.drain_first + i) * N;
        memcpy(dst, ln.pin_out + (size_t)i * N, N * sizeof(float));
    }
    AuxOut o[4], s[4];
    aux_outs(ln.drain_aux, o);
    aux_outs(ln.pin_aux, s);
    for (int k = 0; k < 4; k++)
        if (o[k].p) memcpy(o[k].p + (size_t)ln.drain_first * N * o[k].el, s[k].p, (size_t)ln.drain_n * N * o[k].el);
    ln.drain_aux = adc_aux_outputs{};
    ln.drain_n = 0;
    return ADC_OK;
}

enum SrcKind { SRC_HOST_PTRS, SRC_HOST_STRIDED, SRC_DEVICE_STRIDED };

// Common batch driver.  `user` = stream to fork from / join to.
// `force_join`: the call is one of the synchronous entry points, whose results must be complete on return whatever the
// engine's pipelined setting (adc_set_pipelined only changes the asynchronous entry points).
int run_batch(adc_engine* e, int n, SrcKind kind, const uint8_t* const* lp, const uint8_t* const* rp,
              float* const* dp, const uint8_t* ls, const uint8_t* rs, float* ds, cudaStream_t user, bool pinned,
              bool force_join = false, const adc_aux_outputs* ua = nullptr) {
    const size_t N = (size_t)e->P.dm.N, IMG = N * 3;
    const int S = e->S, nl = (int)e->lanes.size();
    CK(cudaEventRecord(e->ev_fork, user));
    const int n_waves = (n + S - 1) / S;
    for (int li = 0; li < std::min(nl, n_waves); li++) CK(cudaStreamWaitEvent(e->lanes[li].st, e->ev_fork, 0));
    for (int wv = 0; wv < n_waves; wv++) {
        Lane& ln = e->lanes[wv % nl];
        const int first = wv * S, nS = std::min(S, n - first);
        const AdcWave& io = ln.w;   // where the images go in and the map comes out
        // ---- inputs -> io.bgr  ([S][2][IMG])
        if (kind == SRC_DEVICE_STRIDED) {
            CK(cudaMemcpy2DAsync(io.bgr, 2 * IMG, ls + (size_t)first * IMG, IMG, IMG, nS, cudaMemcpyDeviceToDevice, ln.st));
            CK(cudaMemcpy2DAsync(io.bgr + IMG, 2 * IMG, rs + (size_t)first * IMG, IMG, IMG, nS, cudaMemcpyDeviceToDevice, ln.st));
        } else if (pinned) {
            if (kind == SRC_HOST_STRIDED) {
                CK(cudaMemcpy2DAsync(io.bgr, 2 * IMG, ls + (size_t)first * IMG, IMG, IMG, nS, cudaMemcpyHostToDevice, ln.st));
                CK(cudaMemcpy2DAsync(io.bgr + IMG, 2 * IMG, rs + (size_t)first * IMG, IMG, IMG, nS, cudaMemcpyHostToDevice, ln.st));
            } else {
                for (int i = 0; i < nS; i++) {
                    CK(cudaMemcpyAsync(io.bgr + (size_t)i * 2 * IMG, lp[first + i], IMG, cudaMemcpyHostToDevice, ln.st));
                    CK(cudaMemcpyAsync(io.bgr + (size_t)i * 2 * IMG + IMG, rp[first + i], IMG, cudaMemcpyHostToDevice, ln.st));
                }
            }
        } else {
            // pageable caller memory: finish the lane's previous wave (copy-out), then stage through pinned memory
            int rcd = drain_lane(e, ln);
            if (rcd) return rcd;
            CK(cudaEventSynchronize(ln.ev_in_free));
            for (int i = 0; i < nS; i++) {
                const uint8_t* l = kind == SRC_HOST_PTRS ? lp[first + i] : ls + (size_t)(first + i) * IMG;
                const uint8_t* r = kind == SRC_HOST_PTRS ? rp[first + i] : rs + (size_t)(first + i) * IMG;
                memcpy(ln.pin_in + (size_t)i * 2 * IMG, l, IMG);
                memcpy(ln.pin_in + (size_t)i * 2 * IMG + IMG, r, IMG);
            }
            CK(cudaMemcpyAsync(io.bgr, ln.pin_in, (size_t)nS * 2 * IMG, cudaMemcpyHostToDevice, ln.st));
            CK(cudaEventRecord(ln.ev_in_free, ln.st));
        }
        // ---- compute
        cudaStream_t rst = ln.st;   // stream on which the map becomes available
        const AdcAux ax = ua ? wave_aux(ln, *ua) : AdcAux{};
        int rc = enqueue_pipeline(e, ln, nS, ADC_STAGE_MEDIAN, nullptr, ua ? &ax : nullptr);
        if (rc) return rc;
        // ---- outputs
        if (kind == SRC_DEVICE_STRIDED) {
            CK(cudaMemcpyAsync(ds + (size_t)first * N, io.disp_l, (size_t)nS * N * sizeof(float), cudaMemcpyDeviceToDevice, rst));
            if (ua && (rc = copy_aux_out(ln, ax, *ua, first, nS, N, cudaMemcpyDeviceToDevice, rst))) return rc;
        } else if (pinned) {
            if (kind == SRC_HOST_STRIDED) {
                CK(cudaMemcpyAsync(ds + (size_t)first * N, io.disp_l, (size_t)nS * N * sizeof(float), cudaMemcpyDeviceToHost, rst));
                if (ua && (rc = copy_aux_out(ln, ax, *ua, first, nS, N, cudaMemcpyDeviceToHost, rst))) return rc;
            } else {
                for (int i = 0; i < nS; i++)
                    CK(cudaMemcpyAsync(dp[first + i], io.disp_l + (size_t)i * N, N * sizeof(float), cudaMemcpyDeviceToHost, rst));
            }
        } else {
            CK(cudaMemcpyAsync(ln.pin_out, io.disp_l, (size_t)nS * N * sizeof(float), cudaMemcpyDeviceToHost, rst));
            if (ua) {
                if ((rc = copy_aux_out(ln, ax, staging_for(ln, *ua), 0, nS, N, cudaMemcpyDeviceToHost, rst))) return rc;
                ln.drain_aux = *ua;
            }
            ln.drain_n = nS; ln.drain_first = first;
            ln.drain_ptrs = kind == SRC_HOST_PTRS ? dp : nullptr;
            ln.drain_base = ds;
        }
        CK(cudaEventRecord(ln.ev_done, rst));
    }
    // join: the caller's stream waits for every lane -- unless the engine is in pipelined mode, where consecutive
    // batch calls flow into each other (a lane starts the next call's wave while other lanes still finish the
    // previous call's) and the caller joins once with adc_join
    if (!e->pipelined || force_join || (!pinned && kind != SRC_DEVICE_STRIDED))
        for (int li = 0; li < std::min(nl, n_waves); li++) CK(cudaStreamWaitEvent(user, e->lanes[li].ev_done, 0));
    if (!pinned && kind != SRC_DEVICE_STRIDED)
        for (auto& ln : e->lanes) { int rc = drain_lane(e, ln); if (rc) return rc; }
    return ADC_OK;
}

}  // namespace

// =============================================================================================
extern "C" {

const char* adc_last_error(void) { return g_err.c_str(); }
const char* adc_version(void) { return "adcensus_b200 0.1 (sm_100a)"; }

void adc_default_option(adc_option* o) {
    if (!o) return;
    memset(o, 0, sizeof(*o));
    o->min_disparity = 0;  o->max_disparity = 64;
    o->lambda_ad = 10;     o->lambda_census = 30;
    o->cross_L1 = 34;      o->cross_L2 = 17;
    o->cross_t1 = 20;      o->cross_t2 = 6;
    o->so_p1 = 1.0f;       o->so_p2 = 3.0f;
    o->so_tso = 15;        o->irv_ts = 20;
    o->irv_th = 0.4f;      o->lrcheck_thres = 1.0f;
    o->do_lr_check = 1;    o->do_filling = 1;
    o->do_discontinuity_adjustment = 0;
}

void adc_destroy(adc_engine* e) {
    if (!e) return;
    cudaSetDevice(e->cfg.device);
    cudaDeviceSynchronize();
    for (auto& ln : e->lanes) {
        if (ln.arena) cudaFree(ln.arena);
        if (ln.pin_in) cudaFreeHost(ln.pin_in);
        if (ln.pin_out) cudaFreeHost(ln.pin_out);
        if (ln.aux_arena) cudaFree(ln.aux_arena);
        if (ln.aux_pin) cudaFreeHost(ln.aux_pin);
        if (ln.ev_done) cudaEventDestroy(ln.ev_done);
        if (ln.ev_in_free) cudaEventDestroy(ln.ev_in_free);
        if (ln.st) cudaStreamDestroy(ln.st);
    }
    if (e->d_lut_ad) cudaFree(e->d_lut_ad);
    if (e->d_lut_cen) cudaFree(e->d_lut_cen);
    if (e->d_rays) cudaFree(e->d_rays);
    if (e->d_ray_off) cudaFree(e->d_ray_off);
    if (e->ev_fork) cudaEventDestroy(e->ev_fork);
    for (auto& ev : e->ev_stage) if (ev) cudaEventDestroy(ev);
    if (e->main_st) cudaStreamDestroy(e->main_st);
    delete e;
}

int adc_create(int32_t width, int32_t height, const adc_option* opt, const adc_config* cfg, adc_engine** out) {
    if (!out) return fail(ADC_ERR_ARG, "adc_create: out is NULL");
    *out = nullptr;
    if (!opt) return fail(ADC_ERR_ARG, "adc_create: option is NULL");
    if (width <= 0 || height <= 0) return fail(ADC_ERR_ARG, "adc_create: non-positive image size %dx%d", width, height);
    if (opt->max_disparity - opt->min_disparity <= 0)
        return fail(ADC_ERR_ARG, "adc_create: empty disparity range [%d,%d)", opt->min_disparity, opt->max_disparity);
    // Limits of the kernels (the reference has none; INTEGRATION.md lists them).  They are checked HERE, so that a caller
    // never sees Initialize() succeed and Match() fail for a size: whatever adc_create accepts, adc_match runs.
    const int drange = opt->max_disparity - opt->min_disparity;
    const int limit_cfg = cfg ? cfg->max_disparity_range : 0;
    if (limit_cfg < 0 || limit_cfg > ADC_MAX_DISPARITY_RANGE_WIDE)
        return fail(ADC_ERR_ARG, "adc_create: max_disparity_range %d outside 0..%d", limit_cfg, ADC_MAX_DISPARITY_RANGE_WIDE);
    const int limit = limit_cfg ? limit_cfg : ADC_MAX_DISPARITY_RANGE;
    if ((long long)width * height > (1ll << 28)) return fail(ADC_ERR_UNSUPPORTED, "adc_create: image too large (more than 2^28 pixels)");
    if (drange > limit)
        return fail(ADC_ERR_UNSUPPORTED, "adc_create: disparity range %d > %d is not supported by this engine (adc_config.max_disparity_range "
                    "raises the limit up to %d)", drange, limit, ADC_MAX_DISPARITY_RANGE_WIDE);
    if (height > ADC_MAX_HEIGHT)
        return fail(ADC_ERR_UNSUPPORTED, "adc_create: image height %d > %d is not supported (in-place median: one CTA per image)", height, ADC_MAX_HEIGHT);
    if (width > ADC_MAX_WIDTH || width + drange > ADC_MAX_WIDTH)
        return fail(ADC_ERR_UNSUPPORTED, "adc_create: image width %d (+ disparity range %d) > %d is not supported (widest size the kernels are validated for)", width, drange, ADC_MAX_WIDTH);

    adc_engine* e = new adc_engine();
    e->W = width; e->H = height; e->opt = *opt;
    if (cfg) e->cfg = *cfg;
    e->cfg.max_disparity_range = limit;
    build_params(e);
    // kernels whose shared memory grows with the sizes: a launch that could not get its shared memory must fail here
    {
        struct { const char* name; size_t (*need)(const AdcDims&, size_t*); } smem[] = {
            {"cost volume", adc_cost_smem}, {"scanline", adc_scanline_smem}, {"region voting", adc_voting_smem}};
        for (const auto& k : smem) {
            size_t cap = 0;
            const size_t need = k.need(e->P.dm, &cap);
            if (need > cap) {
                delete e;
                return fail(ADC_ERR_UNSUPPORTED, "adc_create: the %s kernel needs %zu bytes of shared memory at %dx%d, disparity "
                            "range %d (at most %zu)", k.name, need, width, height, drange, cap);
            }
        }
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        delete e;
        return fail(ADC_ERR_CUDA, "adc_create: no CUDA device available (this library has no CPU fallback)");
    }
    if (e->cfg.device < 0 || e->cfg.device >= ndev) { delete e; return fail(ADC_ERR_ARG, "adc_create: bad device ordinal"); }
    auto bail = [&](int rc) { adc_destroy(e); return rc; };
    if (cudaSetDevice(e->cfg.device) != cudaSuccess) return bail(fail(ADC_ERR_CUDA, "cudaSetDevice failed"));

    // wave size: enough scanlines in flight for the line-per-lane-group scanline kernels (measured on Cone: 32 pairs
    // per wave x 4 lanes beats 16 x 6; the scanline passes only have W or H lines per pair to spread over 148 SMs)
    int S = e->cfg.wave_pairs;
    if (S <= 0) S = std::min(32, std::max(2, (12288 + std::min(width, height) - 1) / std::min(width, height)));
    int nl = e->cfg.lanes > 0 ? e->cfg.lanes : 4;
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) return bail(fail(ADC_ERR_CUDA, "cudaMemGetInfo failed"));
    while (true) {
        const size_t need = carve_lane(nullptr, e->P.dm, e->P.L1, S, nullptr) * nl;
        if (need < free_b * 8 / 10) break;
        if (nl > 1) nl--; else if (S > 1) S--; else return bail(fail(ADC_ERR_NOMEM, "adc_create: one pair does not fit in device memory"));
    }
    e->S = S;
    e->cfg.wave_pairs = S; e->cfg.lanes = nl;
    e->agg_fused = adc_arm_sum2_available(e->P) && !(e->cfg.debug_flags & ADC_DBG_UNFUSED_AGG);

    int rc = upload_tables(e);
    if (rc) return bail(rc);
    if (cudaStreamCreateWithFlags(&e->main_st, cudaStreamNonBlocking) != cudaSuccess) return bail(fail(ADC_ERR_CUDA, "stream create failed"));
    if (cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming) != cudaSuccess) return bail(fail(ADC_ERR_CUDA, "event create failed"));
    for (auto& ev : e->ev_stage) if (cudaEventCreate(&ev) != cudaSuccess) return bail(fail(ADC_ERR_CUDA, "event create failed"));
    e->lanes.resize(nl);
    const size_t N = (size_t)e->P.dm.N;
    for (auto& ln : e->lanes) {
        if (cudaStreamCreateWithFlags(&ln.st, cudaStreamNonBlocking) != cudaSuccess) return bail(fail(ADC_ERR_CUDA, "stream create failed"));
        if (cudaEventCreateWithFlags(&ln.ev_done, cudaEventDisableTiming) != cudaSuccess) return bail(fail(ADC_ERR_CUDA, "event create failed"));
        if (cudaEventCreateWithFlags(&ln.ev_in_free, cudaEventDisableTiming) != cudaSuccess) return bail(fail(ADC_ERR_CUDA, "event create failed"));
        const size_t bytes = carve_lane(nullptr, e->P.dm, e->P.L1, S, nullptr);
        if (cudaMalloc(&ln.arena, bytes) != cudaSuccess) { cudaGetLastError(); return bail(fail(ADC_ERR_NOMEM, "device arena of %zu bytes", bytes)); }
        carve_lane(ln.arena, e->P.dm, e->P.L1, S, &ln.w);
        if (adc_arm_tmaps_encode(e->P, S, ln.w.volA, ln.w.volB, &ln.arm_tm)) ln.w.arm_tm = &ln.arm_tm;
        if (cudaMemsetAsync(ln.arena, 0, bytes, ln.st) != cudaSuccess) return bail(fail(ADC_ERR_CUDA, "memset failed"));
        if (cudaHostAlloc((void**)&ln.pin_in, (size_t)S * 2 * N * 3, cudaHostAllocDefault) != cudaSuccess ||
            cudaHostAlloc((void**)&ln.pin_out, (size_t)S * N * sizeof(float), cudaHostAllocDefault) != cudaSuccess) {
            cudaGetLastError();
            return bail(fail(ADC_ERR_NOMEM, "pinned staging allocation failed"));
        }
    }
    if (cudaDeviceSynchronize() != cudaSuccess) return bail(fail(ADC_ERR_CUDA, "device sync failed: %s", cudaGetErrorString(cudaGetLastError())));
    *out = e;
    return ADC_OK;
}

}  // extern "C"

namespace {

// One pair on lane 0 through pinned staging: adc_match, and adc_match_aux with `ua` = the wanted side outputs.
int match_one(adc_engine* e, const uint8_t* img_left, const uint8_t* img_right, float* disp_left, const adc_aux_outputs* ua) {
    CK(cudaSetDevice(e->cfg.device));
    Lane& ln = e->lanes[0];
    const size_t N = (size_t)e->P.dm.N, IMG = N * 3;
    int rc = ua ? ensure_aux(e, aux_needs_scratch(ua), 1) : ADC_OK;
    if (rc) return rc;
    if ((rc = drain_lane(e, ln))) return rc;
    CK(cudaStreamSynchronize(ln.st));
    memcpy(ln.pin_in, img_left, IMG);
    memcpy(ln.pin_in + IMG, img_right, IMG);
    CK(cudaEventRecord(e->ev_stage[0], ln.st));
    CK(cudaMemcpyAsync(ln.w.bgr, ln.pin_in, 2 * IMG, cudaMemcpyHostToDevice, ln.st));
    const AdcAux ax = ua ? wave_aux(ln, *ua) : AdcAux{};
    rc = enqueue_pipeline(e, ln, 1, ADC_STAGE_MEDIAN, e->ev_stage, ua ? &ax : nullptr);
    if (rc) return rc;
    CK(cudaMemcpyAsync(ln.pin_out, ln.w.disp_l, N * sizeof(float), cudaMemcpyDeviceToHost, ln.st));
    if (ua && (rc = copy_aux_out(ln, ax, staging_for(ln, *ua), 0, 1, N, cudaMemcpyDeviceToHost, ln.st))) return rc;
    CK(cudaEventRecord(e->ev_stage[6], ln.st));
    CK(cudaStreamSynchronize(ln.st));
    memcpy(disp_left, ln.pin_out, N * sizeof(float));
    if (ua) {
        AuxOut o[4], s[4];
        aux_outs(*ua, o);
        aux_outs(ln.pin_aux, s);
        for (int k = 0; k < 4; k++)
            if (o[k].p) memcpy(o[k].p, s[k].p, N * o[k].el);
    }
    for (int i = 0; i < 6; i++) CK(cudaEventElapsedTime(&e->stage_ms[i], e->ev_stage[i], e->ev_stage[i + 1]));
    return ADC_OK;
}

}  // namespace

extern "C" {

int adc_match(adc_engine* e, const uint8_t* img_left, const uint8_t* img_right, float* disp_left) {
    if (!e) return fail(ADC_ERR_ARG, "adc_match: engine is NULL (Match before Initialize)");
    if (!img_left || !img_right || !disp_left) return fail(ADC_ERR_ARG, "adc_match: NULL image or output pointer");
    return match_one(e, img_left, img_right, disp_left, nullptr);
}

int adc_match_aux(adc_engine* e, const uint8_t* img_left, const uint8_t* img_right, float* disp_left,
                  const adc_aux_outputs* aux) {
    if (!e) return fail(ADC_ERR_ARG, "adc_match_aux: engine is NULL (Match before Initialize)");
    if (!img_left || !img_right || !disp_left) return fail(ADC_ERR_ARG, "adc_match_aux: NULL image or output pointer");
    return match_one(e, img_left, img_right, disp_left, aux_wanted(aux) ? aux : nullptr);
}

int adc_get_right_disparity(adc_engine* e, float* disp_right) {
    if (!e || !disp_right) return fail(ADC_ERR_ARG, "adc_get_right_disparity: bad arguments");
    CK(cudaSetDevice(e->cfg.device));
    Lane& ln = e->lanes[0];
    CK(cudaStreamSynchronize(ln.st));
    CK(cudaMemcpy(disp_right, ln.w.disp_r, (size_t)e->P.dm.N * sizeof(float), cudaMemcpyDeviceToHost));
    return ADC_OK;
}

int adc_match_batch(adc_engine* e, int32_t n, const uint8_t* const* img_left, const uint8_t* const* img_right,
                    float* const* disp_left) {
    if (!e) return fail(ADC_ERR_ARG, "adc_match_batch: engine is NULL");
    if (n < 0 || (n > 0 && (!img_left || !img_right || !disp_left))) return fail(ADC_ERR_ARG, "adc_match_batch: bad arguments");
    if (n == 0) return ADC_OK;
    bool pinned = true;
    for (int i = 0; i < n; i++) {
        if (!img_left[i] || !img_right[i] || !disp_left[i]) return fail(ADC_ERR_ARG, "adc_match_batch: NULL pointer for pair %d", i);
    }
    CK(cudaSetDevice(e->cfg.device));
    for (int i = 0; i < n && pinned; i++) pinned = is_pinned(img_left[i]) && is_pinned(img_right[i]) && is_pinned(disp_left[i]);
    int rc = run_batch(e, n, SRC_HOST_PTRS, img_left, img_right, disp_left, nullptr, nullptr, nullptr, e->main_st, pinned, true);
    if (rc) return rc;
    CK(cudaStreamSynchronize(e->main_st));
    return ADC_OK;
}

int adc_match_batch_strided(adc_engine* e, int32_t n, const uint8_t* left, const uint8_t* right, float* disp) {
    if (!e) return fail(ADC_ERR_ARG, "adc_match_batch_strided: engine is NULL");
    if (n < 0 || (n > 0 && (!left || !right || !disp))) return fail(ADC_ERR_ARG, "adc_match_batch_strided: bad arguments");
    if (n == 0) return ADC_OK;
    CK(cudaSetDevice(e->cfg.device));
    const bool pinned = is_pinned(left) && is_pinned(right) && is_pinned(disp);
    int rc = run_batch(e, n, SRC_HOST_STRIDED, nullptr, nullptr, nullptr, left, right, disp, e->main_st, pinned, true);
    if (rc) return rc;
    CK(cudaStreamSynchronize(e->main_st));
    return ADC_OK;
}

int adc_match_batch_strided_aux(adc_engine* e, int32_t n, const uint8_t* left, const uint8_t* right, float* disp,
                                const adc_aux_outputs* aux) {
    if (!e) return fail(ADC_ERR_ARG, "adc_match_batch_strided_aux: engine is NULL");
    if (n < 0 || (n > 0 && (!left || !right || !disp))) return fail(ADC_ERR_ARG, "adc_match_batch_strided_aux: bad arguments");
    if (n == 0) return ADC_OK;
    const adc_aux_outputs* ua = aux_wanted(aux) ? aux : nullptr;
    CK(cudaSetDevice(e->cfg.device));
    bool pinned = is_pinned(left) && is_pinned(right) && is_pinned(disp);
    if (ua) {
        AuxOut o[4];
        aux_outs(*ua, o);
        for (int k = 0; k < 4; k++) pinned = pinned && (!o[k].p || is_pinned(o[k].p));
        int rc = ensure_aux(e, aux_needs_scratch(ua), pinned ? 0 : (int)e->lanes.size());
        if (rc) return rc;
    }
    int rc = run_batch(e, n, SRC_HOST_STRIDED, nullptr, nullptr, nullptr, left, right, disp, e->main_st, pinned, true, ua);
    if (rc) return rc;
    CK(cudaStreamSynchronize(e->main_st));
    return ADC_OK;
}

int adc_match_batch_pinned_async(adc_engine* e, int32_t n, const uint8_t* left, const uint8_t* right, float* disp, void* stream) {
    if (!e) return fail(ADC_ERR_ARG, "adc_match_batch_pinned_async: engine is NULL");
    if (n < 0 || (n > 0 && (!left || !right || !disp))) return fail(ADC_ERR_ARG, "adc_match_batch_pinned_async: bad arguments");
    if (n == 0) return ADC_OK;
    CK(cudaSetDevice(e->cfg.device));
    if (!(is_pinned(left) && is_pinned(right) && is_pinned(disp)))
        return fail(ADC_ERR_ARG, "adc_match_batch_pinned_async: buffers must be pinned host memory");
    return run_batch(e, n, SRC_HOST_STRIDED, nullptr, nullptr, nullptr, left, right, disp, (cudaStream_t)stream, true);
}

int adc_match_batch_device(adc_engine* e, int32_t n, const uint8_t* d_left, const uint8_t* d_right, float* d_disp, void* stream) {
    if (!e) return fail(ADC_ERR_ARG, "adc_match_batch_device: engine is NULL");
    if (n < 0 || (n > 0 && (!d_left || !d_right || !d_disp))) return fail(ADC_ERR_ARG, "adc_match_batch_device: bad arguments");
    if (n == 0) return ADC_OK;
    CK(cudaSetDevice(e->cfg.device));
    return run_batch(e, n, SRC_DEVICE_STRIDED, nullptr, nullptr, nullptr, d_left, d_right, d_disp, (cudaStream_t)stream, true);
}

int adc_match_batch_device_aux(adc_engine* e, int32_t n, const uint8_t* d_left, const uint8_t* d_right, float* d_disp,
                               const adc_aux_outputs* aux, void* stream) {
    if (!e) return fail(ADC_ERR_ARG, "adc_match_batch_device_aux: engine is NULL");
    if (n < 0 || (n > 0 && (!d_left || !d_right || !d_disp))) return fail(ADC_ERR_ARG, "adc_match_batch_device_aux: bad arguments");
    if (n == 0) return ADC_OK;
    const adc_aux_outputs* ua = aux_wanted(aux) ? aux : nullptr;
    CK(cudaSetDevice(e->cfg.device));
    if (ua) {
        int rc = ensure_aux(e, aux_needs_scratch(ua), 0);
        if (rc) return rc;
    }
    return run_batch(e, n, SRC_DEVICE_STRIDED, nullptr, nullptr, nullptr, d_left, d_right, d_disp, (cudaStream_t)stream, true,
                     false, ua);
}

void* adc_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
void adc_host_free(void* p) { if (p) cudaFreeHost(p); }

int adc_synchronize(adc_engine* e) {
    if (!e) return fail(ADC_ERR_ARG, "adc_synchronize: engine is NULL");
    CK(cudaSetDevice(e->cfg.device));
    for (auto& ln : e->lanes) {
        CK(cudaStreamSynchronize(ln.st));
    }
    CK(cudaStreamSynchronize(e->main_st));
    return ADC_OK;
}

int adc_set_pipelined(adc_engine* e, int32_t on) {
    if (!e) return fail(ADC_ERR_ARG, "adc_set_pipelined: engine is NULL");
    e->pipelined = on != 0;
    return ADC_OK;
}

int adc_join(adc_engine* e, void* stream) {
    if (!e) return fail(ADC_ERR_ARG, "adc_join: engine is NULL");
    CK(cudaSetDevice(e->cfg.device));
    for (auto& ln : e->lanes) CK(cudaStreamWaitEvent((cudaStream_t)stream, ln.ev_done, 0));
    return ADC_OK;
}

uint64_t adc_launch_count(const adc_engine* e) { return e ? e->launches : 0; }

int adc_last_stage_ms(const adc_engine* e, float out[6]) {
    if (!e || !out) return fail(ADC_ERR_ARG, "adc_last_stage_ms: bad arguments");
    // ev_stage[0..6]: start | cost | aggregation | scanline | wta | refine | output copy
    for (int i = 0; i < 6; i++) out[i] = e->stage_ms[i];
    return ADC_OK;
}

int adc_get_config(const adc_engine* e, adc_config* out) {
    if (!e || !out) return fail(ADC_ERR_ARG, "adc_get_config: bad arguments");
    *out = e->cfg;
    return ADC_OK;
}

// ---- output side of the reference's demo (main.cpp:147-230), SURVEY.md 8(f) rank 3 ----------------------------
int adc_render_disparity(adc_engine* e, const float* disp, uint8_t* gray8, uint8_t* jet_bgr, float* min_max) {
    if (!e) return fail(ADC_ERR_ARG, "adc_render_disparity: engine is NULL");
    if (!disp || (!gray8 && !jet_bgr && !min_max)) return fail(ADC_ERR_ARG, "adc_render_disparity: NULL map or no output requested");
    CK(cudaSetDevice(e->cfg.device));
    Lane& ln = e->lanes[0];
    int rc = drain_lane(e, ln);
    if (rc) return rc;
    CK(cudaStreamSynchronize(ln.st));
    const size_t N = (size_t)e->P.dm.N;
    // lane 0's buffers are idle between calls: disp_t holds the map, flag the 8-bit image, bgr the colour image,
    // the first words of tile_stamp the min/max keys and (as floats) the values handed back
    float* d_disp = ln.w.disp_t;
    unsigned* d_mm = reinterpret_cast<unsigned*>(ln.w.rowcnt);
    float* d_mm_out = reinterpret_cast<float*>(ln.w.rowcnt) + 2;
    CK(cudaMemcpyAsync(d_disp, disp, N * sizeof(float), cudaMemcpyHostToDevice, ln.st));
    if (adc_launch_render(e->P.dm, d_disp, d_mm, ln.w.flag, ln.w.bgr, d_mm_out, ln.st, &e->launches))
        return fail(ADC_ERR_CUDA, "adc_render_disparity: colour table upload failed");
    if (gray8) CK(cudaMemcpyAsync(gray8, ln.w.flag, N, cudaMemcpyDeviceToHost, ln.st));
    if (jet_bgr) CK(cudaMemcpyAsync(jet_bgr, ln.w.bgr, 3 * N, cudaMemcpyDeviceToHost, ln.st));
    if (min_max) CK(cudaMemcpyAsync(min_max, d_mm_out, 2 * sizeof(float), cudaMemcpyDeviceToHost, ln.st));
    CK(cudaStreamSynchronize(ln.st));
    CK(cudaGetLastError());
    return ADC_OK;
}

int adc_disparity_cloud(adc_engine* e, const uint8_t* img_left, const float* disp, float* cloud, int32_t* n_points) {
    if (!e) return fail(ADC_ERR_ARG, "adc_disparity_cloud: engine is NULL");
    if (!img_left || !disp || !cloud || !n_points) return fail(ADC_ERR_ARG, "adc_disparity_cloud: NULL pointer");
    CK(cudaSetDevice(e->cfg.device));
    Lane& ln = e->lanes[0];
    int rc = drain_lane(e, ln);
    if (rc) return rc;
    CK(cudaStreamSynchronize(ln.st));
    const size_t N = (size_t)e->P.dm.N;
    const AdcWave w1 = wave_view(e, ln, 1);
    float* d_cloud = ln.w.volA;                       // 6 floats per pixel at most; a volume has Dp >= 4 ... use both volumes' span
    if ((size_t)e->P.dm.vol_stride * 2 < N * 6) return fail(ADC_ERR_UNSUPPORTED, "adc_disparity_cloud: disparity range too small for the scratch volume");
    CK(cudaMemcpyAsync(ln.w.disp_t, disp, N * sizeof(float), cudaMemcpyHostToDevice, ln.st));
    CK(cudaMemcpyAsync(ln.w.bgr, img_left, 3 * N, cudaMemcpyHostToDevice, ln.st));
    CK(cudaMemsetAsync(ln.w.counters, 0, ADC_CNT * sizeof(int), ln.st));
    adc_launch_cloud(e->P, w1, ln.w.disp_t, ln.w.bgr, d_cloud, ln.st, &e->launches);
    int n = 0;
    CK(cudaMemcpyAsync(&n, ln.w.counters, sizeof(int), cudaMemcpyDeviceToHost, ln.st));
    CK(cudaStreamSynchronize(ln.st));
    if (n > 0) CK(cudaMemcpy(cloud, d_cloud, (size_t)n * 6 * sizeof(float), cudaMemcpyDeviceToHost));
    *n_points = n;
    CK(cudaGetLastError());
    return ADC_OK;
}

// ---- per-kernel timing for the roofline figures of bench.py ------------------------------------
// Re-launches ONE kernel of the pipeline `reps` times on lane 0's wave buffers (which hold whatever
// the last batch left there; every kernel below is data-oblivious in its memory traffic except for
// the arm lengths, which are real) and reports the mean device time per launch, measured with CUDA
// events on the lane's own stream, plus the algorithmic bytes one launch moves (SURVEY.md 8d model).
int adc_profile_kernel(adc_engine* e, int32_t kernel_id, int32_t reps, float* avg_ms, double* algorithmic_bytes) {
    if (!e || !avg_ms || reps <= 0) return fail(ADC_ERR_ARG, "adc_profile_kernel: bad arguments");
    CK(cudaSetDevice(e->cfg.device));
    Lane& ln = e->lanes[0];
    const AdcParams& P = e->P;
    const AdcWave w = wave_view(e, ln, e->S);
    const double V = (double)P.dm.N * P.dm.D * 4.0, N = (double)P.dm.N;
    double bytes = 0;
    CK(cudaStreamSynchronize(ln.st));
    cudaEvent_t e0 = e->ev_stage[0], e1 = e->ev_stage[1];
    for (int r = -1; r < reps; r++) {   // r = -1: warm-up launch
        if (r == 0) CK(cudaEventRecord(e0, ln.st));
        switch (kernel_id) {
            case 0: adc_launch_cost(P, w, w.volB, ln.st, &e->launches); bytes = V + 6 * N + 16 * N; break;
            case 1: adc_launch_arm_sum(P, w, w.volA, w.volB, 0, nullptr, ln.st, &e->launches); bytes = 2 * V + 4 * N; break;
            case 2: adc_launch_arm_sum(P, w, w.volA, w.volB, 1, w.sup_h, ln.st, &e->launches); bytes = 2 * V + 6 * N; break;
            case 3: if (adc_launch_scanline(P, w, w.volA, w.volB, 1, 0, ln.st, &e->launches)) return fail(ADC_ERR_UNSUPPORTED, "scanline"); bytes = 2 * V + 6 * N; break;
            case 4: if (adc_launch_scanline(P, w, w.volA, w.volB, 0, 1, ln.st, &e->launches)) return fail(ADC_ERR_UNSUPPORTED, "scanline"); bytes = 2 * V + 6 * N; break;
            case 5: if (adc_launch_wta(P, w, w.volA, ln.st, &e->launches)) return fail(ADC_ERR_UNSUPPORTED, "wta"); bytes = V + 8 * N; break;
            case 6: if (!adc_launch_arm_sum2(P, w, w.volA, w.volB, 1, w.sup_h, ln.st, &e->launches)) return fail(ADC_ERR_UNSUPPORTED, "fused vertical arm sums not applicable"); bytes = 2 * V + 6 * N; break;
            case 7: if (!adc_launch_arm_sum2(P, w, w.volA, w.volB, 0, w.sup_v, ln.st, &e->launches)) return fail(ADC_ERR_UNSUPPORTED, "fused horizontal arm sums not applicable"); bytes = 2 * V + 6 * N; break;
            case 8: adc_launch_arm_sum(P, w, w.volA, w.volB, 0, w.sup_v, ln.st, &e->launches); bytes = 2 * V + 6 * N; break;
            case 9: adc_launch_arm_sum(P, w, w.volA, w.volB, 1, nullptr, ln.st, &e->launches); bytes = 2 * V + 4 * N; break;
            case 10: {
                int rc = ensure_aux(e, true, 0);
                if (rc) return rc;
                const AdcAux ax{ln.aux.origin, nullptr, ln.aux.cost_best, ln.aux.cost_second};
                if (adc_launch_wta_aux(P, w, w.volA, ax, ln.st, &e->launches)) return fail(ADC_ERR_UNSUPPORTED, "wta");
                bytes = V + 17 * N;
                break;
            }
            default: return fail(ADC_ERR_ARG, "adc_profile_kernel: unknown kernel id %d", kernel_id);
        }
    }
    CK(cudaEventRecord(e1, ln.st));
    CK(cudaStreamSynchronize(ln.st));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    *avg_ms = ms / reps;
    if (algorithmic_bytes) *algorithmic_bytes = bytes * e->S;
    return ADC_OK;
}

// ---- debug taps -----------------------------------------------------------------------------
int adc_debug_run(adc_engine* e, const uint8_t* img_left, const uint8_t* img_right, int32_t last_stage) {
    if (!e) return fail(ADC_ERR_ARG, "adc_debug_run: engine is NULL");
    if (!img_left || !img_right) return fail(ADC_ERR_ARG, "adc_debug_run: NULL image");
    if (last_stage < 0 || last_stage >= ADC_STAGE_COUNT) return fail(ADC_ERR_ARG, "adc_debug_run: bad stage");
    CK(cudaSetDevice(e->cfg.device));
    Lane& ln = e->lanes[0];
    const size_t IMG = (size_t)e->P.dm.N * 3;
    int rc = drain_lane(e, ln);
    if (rc) return rc;
    CK(cudaStreamSynchronize(ln.st));
    CK(cudaMemcpyAsync(ln.w.bgr, img_left, IMG, cudaMemcpyHostToDevice, ln.st));
    CK(cudaMemcpyAsync(ln.w.bgr + IMG, img_right, IMG, cudaMemcpyHostToDevice, ln.st));
    rc = enqueue_pipeline(e, ln, 1, last_stage, nullptr);
    if (rc) return rc;
    CK(cudaStreamSynchronize(ln.st));
    CK(cudaGetLastError());
    return ADC_OK;
}

int adc_debug_counters(adc_engine* e, int32_t out[16]) {
    if (!e || !out) return fail(ADC_ERR_ARG, "adc_debug_counters: bad arguments");
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaMemcpy(out, e->lanes[0].w.counters, 16 * sizeof(int32_t), cudaMemcpyDeviceToHost));
    return ADC_OK;
}

size_t adc_debug_get(adc_engine* e, int32_t tap, void* dst, size_t cap) {
    if (!e) { fail(ADC_ERR_ARG, "adc_debug_get: engine is NULL"); return 0; }
    if (cudaSetDevice(e->cfg.device) != cudaSuccess) return 0;
    const AdcDims& dm = e->P.dm;
    const Lane& ln = e->lanes[0];
    const size_t N = (size_t)dm.N;
    const void* src = nullptr;
    size_t bytes = 0;
    switch (tap) {
        case ADC_TAP_GRAY_L: src = ln.w.gray; bytes = N; break;
        case ADC_TAP_GRAY_R: src = ln.w.gray + N; bytes = N; break;
        case ADC_TAP_CENSUS_L: src = ln.w.census; bytes = N * 8; break;
        case ADC_TAP_CENSUS_R: src = ln.w.census + N; bytes = N * 8; break;
        case ADC_TAP_ARMS: src = ln.w.arms; bytes = N * 4; break;
        case ADC_TAP_SUPCNT_H: src = ln.w.sup_h; bytes = N * 2; break;
        case ADC_TAP_SUPCNT_V: src = ln.w.sup_v; bytes = N * 2; break;
        case ADC_TAP_DISP_L: src = ln.w.disp_l; bytes = N * 4; break;
        case ADC_TAP_DISP_R: src = ln.w.disp_r; bytes = N * 4; break;
        case ADC_TAP_VOL_INIT:
        case ADC_TAP_VOL_AGGR: {
            const float* v = tap == ADC_TAP_VOL_INIT ? e->dbg_init : e->dbg_aggr;
            bytes = N * dm.D * sizeof(float);
            if (!dst || cap < bytes || !v) return bytes;
            // strip the Dp padding: [N][Dp] -> [N][D]
            if (cudaMemcpy2D(dst, (size_t)dm.D * 4, v, (size_t)dm.Dp * 4, (size_t)dm.D * 4, N, cudaMemcpyDeviceToHost) != cudaSuccess) {
                fail(ADC_ERR_CUDA, "adc_debug_get: copy failed: %s", cudaGetErrorString(cudaGetLastError()));
                return 0;
            }
            return bytes;
        }
        case ADC_TAP_MISMATCHES:
        case ADC_TAP_OCCLUSIONS: {
            // the lists are the pixels labelled 1 / 2, in raster order (the reference builds them by a
            // raster scan and only ever erases from them)
            std::vector<uint8_t> lab(N);
            if (cudaMemcpy(lab.data(), ln.w.label, N, cudaMemcpyDeviceToHost) != cudaSuccess) return 0;
            const uint8_t want = tap == ADC_TAP_MISMATCHES ? 1 : 2;
            size_t cnt = 0;
            for (size_t i = 0; i < N; i++) cnt += lab[i] == want;
            bytes = cnt * 8;
            if (!dst || cap < bytes) return bytes;
            int32_t* o = static_cast<int32_t*>(dst);
            for (size_t i = 0; i < N; i++)
                if (lab[i] == want) { *o++ = (int32_t)(i % dm.W); *o++ = (int32_t)(i / dm.W); }
            return bytes;
        }
        default: fail(ADC_ERR_ARG, "adc_debug_get: unknown tap %d", tap); return 0;
    }
    if (!dst || cap < bytes) return bytes;
    if (cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost) != cudaSuccess) {
        fail(ADC_ERR_CUDA, "adc_debug_get: copy failed: %s", cudaGetErrorString(cudaGetLastError()));
        return 0;
    }
    return bytes;
}

}  // extern "C"
