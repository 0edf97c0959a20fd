// k_refine.cu -- stage 5: multi-step disparity refinement (reference: multistep_refiner.cpp:60-87):
// LR-check outlier detection (:90-151), iterative region voting (:153-227), 16-ray proper
// interpolation (:229-305), optional depth-discontinuity adjustment (:307-371) and the in-place 3x3
// median (adcensus_util.cpp:55-81 called with in == out at multistep_refiner.cpp:86).
//
// The reference runs all of these sequentially *in place*, and the in-place order is part of the
// answer.  Each kernel below is a parallel schedule that provably reproduces the sequential
// result (argument given at each kernel); none of them approximates.
#include "adc_common.cuh"
#include "../../include/adcensus_b200.h"
#include <stdlib.h>
#include <algorithm>

// barrier over all threads of the thread-block cluster, with release/acquire ordering of memory
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}

// =============================================================================================
// 1. Outlier detection.  The raster scan reads disp_left[col_rl] of the same row while already
//    having invalidated pixels to the left of x.  Whether a pixel gets invalidated depends only on
//    the ORIGINAL maps (its own disparity and the right map), so: phase 1 computes that predicate
//    for every pixel; phase 2 classifies, seeing +inf for col_rl < x that phase 1 marked, and the
//    original value otherwise (col_rl == x reads the pixel itself before it is invalidated).
// =============================================================================================
__global__ void k_outlier_mark(AdcParams P, const float* __restrict__ disp_l, const float* __restrict__ disp_r,
                               uint8_t* __restrict__ flag) {
    const AdcDims& dm = P.dm;
    const int pair = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= dm.N) return;
    const int y = i / dm.W, x = i - y * dm.W;
    const float d = disp_l[(size_t)pair * dm.N + i];
    uint8_t f = 0;
    if (d == ADC_INVALID_F) f = 1;
    else {
        const long col_r = lroundf(__fsub_rn((float)x, d));
        if (col_r < 0 || col_r >= dm.W) f = 1;
        else {
            const float dr = disp_r[(size_t)pair * dm.N + y * dm.W + col_r];
            if (fabsf(__fsub_rn(d, dr)) > P.lr_thres) f = 2;
        }
    }
    flag[(size_t)pair * dm.N + i] = f;
}

__global__ void k_outlier_classify(AdcParams P, const float* __restrict__ disp_l, const float* __restrict__ disp_r,
                                   const uint8_t* __restrict__ flag, float* __restrict__ disp_out,
                                   uint8_t* __restrict__ label) {
    const AdcDims& dm = P.dm;
    const int pair = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= dm.N) return;
    const size_t o = (size_t)pair * dm.N;
    const int y = i / dm.W, x = i - y * dm.W;
    const uint8_t f = flag[o + i];
    const float d = disp_l[o + i];
    uint8_t lab = 0;
    if (f == 1) lab = 1;
    else if (f == 2) {
        const long col_r = lroundf(__fsub_rn((float)x, d));
        const float dr = disp_r[o + y * dm.W + col_r];
        const int col_rl = (int)lroundf(__fadd_rn((float)col_r, dr));
        lab = 1;
        if (col_rl > 0 && col_rl < dm.W) {
            const int j = y * dm.W + col_rl;
            const float dl = (col_rl < x && flag[o + j] != 0) ? ADC_INVALID_F : disp_l[o + j];
            if (dl > d) lab = 2;
        }
    }
    label[o + i] = lab;
    disp_out[o + i] = f ? ADC_INVALID_F : d;
}

void adc_launch_outlier(const AdcParams& P, const AdcWave& w, cudaStream_t st, unsigned long long* launches) {
    dim3 grid((P.dm.N + 255) / 256, w.S);
    k_outlier_mark<<<grid, 256, 0, st>>>(P, w.disp_l, w.disp_r, w.flag);
    k_outlier_classify<<<grid, 256, 0, st>>>(P, w.disp_l, w.disp_r, w.flag, w.disp_t, w.label);
    *launches += 2;
}

// =============================================================================================
// 2. Iterative region voting -- the PULL form.  The default path is the incremental-histogram (push) form in
//    k_vote.cu; the kernels below remain as the fallback for configurations that path does not take (more than
//    254 disparities, arms longer than 127) and as the A/B reference (ADC_VOTE_MODE=1 / 2 / 3).
//    Reference: 5 iterations x {mismatch list, occlusion list}; within a
//    sweep pixels are visited in list (= raster) order and a filled pixel is immediately visible to
//    later ones (Gauss-Seidel).  Exact parallel form ("raster-aware fixed point"): keep OLD (state at
//    sweep start) and NEW.  Repeatedly recompute pending pixels p of the list in parallel, reading
//    neighbour q from NEW if q precedes p in raster order and from OLD otherwise, until a full round
//    changes nothing.  The sequential result is the unique fixed point of that map (induction over
//    raster order: the first pending pixel only depends on OLD, pixel p only on OLD and on earlier
//    pixels), so ANY asynchronous evaluation order converges to it, and a round without changes
//    certifies it.
//    Work filter (does not change the fixed point): a pixel's vote is a pure function of the
//    disparities inside its cross region, which lies within +-L1 of it.  Every value change stamps
//    the 16x16 tiles within that reach with the current epoch; a pending pixel is re-evaluated only
//    if its tile carries a stamp >= the epoch of its own last evaluation.  Otherwise its inputs are
//    bit-for-bit what they were and so is its vote -- this also carries over from sweep to sweep.
//    One CTA per stereo pair (so plain L1-cached accesses are coherent); the batch and the other
//    lanes keep the rest of the chip busy.
// =============================================================================================
#define RV_THREADS 1024
#define RV_WARPS (RV_THREADS / 32)
#define RV_MAXD 256     // histogram bins of the byte-state kernel (D <= 254); the float-state kernel sizes its own
#define RV_TILE 16

// ---- ordered (raster) pixel lists of the two outlier classes: row counts -> scan -> scatter ----
__global__ void __launch_bounds__(128)
k_list_row_counts(AdcDims dm, const uint8_t* __restrict__ label, const uint16_t* __restrict__ region_size, int min_size,
                  int* __restrict__ rowcnt) {
    // region_size != NULL: only pixels whose cross region holds more than min_size pixels (see adc_launch_voting)
    const int pair = blockIdx.y, y = blockIdx.x;
    const uint8_t* lab = label + (size_t)pair * dm.N + (size_t)y * dm.W;
    const uint16_t* rs = region_size ? region_size + (size_t)pair * dm.N + (size_t)y * dm.W : nullptr;
    int c1 = 0, c2 = 0;
    for (int x = threadIdx.x; x < dm.W; x += 128) {
        uint8_t v = lab[x];
        if (rs && (int)rs[x] <= min_size) v = 0;
        c1 += v == 1; c2 += v == 2;
    }
    __shared__ int s1[4], s2[4];
    c1 = __reduce_add_sync(0xffffffffu, c1);
    c2 = __reduce_add_sync(0xffffffffu, c2);
    if ((threadIdx.x & 31) == 0) { s1[threadIdx.x >> 5] = c1; s2[threadIdx.x >> 5] = c2; }
    __syncthreads();
    if (threadIdx.x == 0) {
        rowcnt[((size_t)pair * 2 + 0) * dm.H + y] = s1[0] + s1[1] + s1[2] + s1[3];
        rowcnt[((size_t)pair * 2 + 1) * dm.H + y] = s2[0] + s2[1] + s2[2] + s2[3];
    }
}

// exclusive scan of the row counts (in place), one warp per (pair, class)
__global__ void __launch_bounds__(64)
k_list_row_scan(AdcDims dm, int* __restrict__ rowcnt, int* __restrict__ counters, int slot) {
    const int pair = blockIdx.x, k = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int* rc = rowcnt + ((size_t)pair * 2 + k) * dm.H;
    int base = 0;
    for (int y0 = 0; y0 < dm.H; y0 += 32) {
        const int y = y0 + lane;
        const int v = y < dm.H ? rc[y] : 0;
        int inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
        if (y < dm.H) rc[y] = base + inc - v;
        base += __shfl_sync(0xffffffffu, inc, 31);
    }
    if (lane == 0) counters[pair * ADC_CNT + slot + k] = base;
}

__global__ void __launch_bounds__(128)
k_list_row_scatter(AdcDims dm, const uint8_t* __restrict__ label, const uint16_t* __restrict__ region_size, int min_size,
                   const int* __restrict__ rowoff, int* __restrict__ pend) {
    const int pair = blockIdx.y, y = blockIdx.x;
    const uint8_t* lab = label + (size_t)pair * dm.N + (size_t)y * dm.W;
    const uint16_t* rs = region_size ? region_size + (size_t)pair * dm.N + (size_t)y * dm.W : nullptr;
    __shared__ int s_cnt[2][4];
    int base1 = rowoff[((size_t)pair * 2 + 0) * dm.H + y], base2 = rowoff[((size_t)pair * 2 + 1) * dm.H + y];
    int* l1 = pend + ((size_t)pair * 2 + 0) * dm.N;
    int* l2 = pend + ((size_t)pair * 2 + 1) * dm.N;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int x0 = 0; x0 < dm.W; x0 += 128) {
        const int x = x0 + threadIdx.x;
        uint8_t v = x < dm.W ? lab[x] : 0;
        if (rs && x < dm.W && (int)rs[x] <= min_size) v = 0;
        const unsigned b1 = __ballot_sync(0xffffffffu, v == 1), b2 = __ballot_sync(0xffffffffu, v == 2);
        if (lane == 0) { s_cnt[0][wid] = __popc(b1); s_cnt[1][wid] = __popc(b2); }
        __syncthreads();
        int o1 = base1, o2 = base2, t1 = 0, t2 = 0;
#pragma unroll
        for (int w2 = 0; w2 < 4; w2++) {
            if (w2 < wid) { o1 += s_cnt[0][w2]; o2 += s_cnt[1][w2]; }
            t1 += s_cnt[0][w2]; t2 += s_cnt[1][w2];
        }
        const unsigned lt = (1u << lane) - 1u;
        if (v == 1) l1[o1 + __popc(b1 & lt)] = y * dm.W + x;
        if (v == 2) l2[o2 + __popc(b2 & lt)] = y * dm.W + x;
        base1 += t1; base2 += t2;
        __syncthreads();
    }
}

void adc_launch_build_lists(const AdcParams& P, const AdcWave& w, cudaStream_t st, unsigned long long* launches) {
    dim3 grid(P.dm.H, w.S);
    k_list_row_counts<<<grid, 128, 0, st>>>(P.dm, w.label, nullptr, 0, w.rowcnt);
    k_list_row_scan<<<w.S, 64, 0, st>>>(P.dm, w.rowcnt, w.counters, 0);
    k_list_row_scatter<<<grid, 128, 0, st>>>(P.dm, w.label, nullptr, 0, w.rowcnt, w.pend);
    *launches += 3;
}

// Lists of the pixels that can still be filled by voting: a vote needs more than irv_ts valid pixels in
// the pixel's cross region (multistep_refiner.cpp:211), and that region -- the vertical arm of p, then the
// horizontal arm of every pixel on it -- is exactly the horizontal-first support region whose size
// cross_aggregator.cpp:271-325 already counted.  A pixel whose whole region is not larger than irv_ts can
// never pass, in any sweep, whatever its neighbours become: it is left out of the voting lists (about 40 %
// of the listed pixels on Cone) and simply stays in the outlier lists for the interpolation step.
static void launch_active_lists(const AdcParams& P, const AdcWave& w, cudaStream_t st, unsigned long long* launches) {
    const bool exact = P.L1 <= 127;   // beyond that the reference's uint16 counts may wrap
    dim3 grid(P.dm.H, w.S);
    k_list_row_counts<<<grid, 128, 0, st>>>(P.dm, w.label, exact ? w.sup_h : nullptr, P.irv_ts, w.rowcnt);
    k_list_row_scan<<<w.S, 64, 0, st>>>(P.dm, w.rowcnt, w.counters, 10);
    k_list_row_scatter<<<grid, 128, 0, st>>>(P.dm, w.label, exact ? w.sup_h : nullptr, P.irv_ts, w.rowcnt, w.vlist);
    *launches += 3;
}

// in-place ordered compaction of list[0..n) keeping the pixels that are still invalid (one CTA)
__device__ int rv_compact_invalid(int n, int* list, const float* d_old, int* s_warp_tot) {
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    int base = 0;
    for (int start = 0; start < n; start += RV_THREADS) {
        const int i = start + tid;
        int p = 0;
        bool keep = false;
        if (i < n) { p = __ldcg(list + i); keep = __ldcg(d_old + p) == ADC_INVALID_F; }
        const unsigned b = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) s_warp_tot[wid] = __popc(b);
        __syncthreads();  // also orders this chunk's reads before its writes
        int off = base, tot = 0;
        for (int w2 = 0; w2 < RV_WARPS; w2++) {
            const int c = s_warp_tot[w2];
            if (w2 < wid) off += c;
            tot += c;
        }
        if (keep) __stcg(list + off + __popc(b & ((1u << lane) - 1u)), p);
        base += tot;
        __syncthreads();
    }
    return base;
}

// `reach_up`: how far above (x,y) dependants can sit.  At commit time that is `reach` (everybody around sees
// the new OLD value); during the rounds of a sweep it is 0: a changed NEW value is only read by pixels that
// come LATER in raster order, and every pixel of a tile row above (x,y)'s own comes earlier.
__device__ __forceinline__ void rv_stamp_tiles(int* tiles, int tw, int th, int x, int y, int reach, int epoch, int lane,
                                               int reach_up) {
    const int tx0 = max(0, (x - reach) / RV_TILE), tx1 = min(tw - 1, (x + reach) / RV_TILE);
    const int ty0 = max(0, (y - reach_up) / RV_TILE), ty1 = min(th - 1, (y + reach) / RV_TILE);
    const int nx = tx1 - tx0 + 1, nt = nx * (ty1 - ty0 + 1);
    for (int i = lane; i < nt; i += 32) __stcg(tiles + (ty0 + i / nx) * tw + tx0 + i % nx, epoch);
}

// A thread-block cluster of RV_CLUSTER CTAs works on one stereo pair: the pending pixels of a
// round are dealt round-robin to its RV_CLUSTER*32 warps, the rounds are separated by cluster
// barriers, and all mutable state lives in global memory and is accessed at L2 (ld.cg / st.cg)
// because the CTAs sit on different SMs.
#define RV_CLUSTER 8

// USE_L1: read through L1 (plain loads).  The cluster barrier between rounds carries an acquire at
// cluster scope, for which ptxas emits an L1 invalidate, so a round never sees lines cached before
// the previous barrier; lines going stale *within* a round are harmless (asynchronous fixed point,
// and the certifying round has no writes at all).
template <bool USE_L1> __device__ __forceinline__ float rv_ld(const float* p) { return USE_L1 ? __ldca(p) : __ldcg(p); }
template <bool USE_L1> __device__ __forceinline__ int rv_ld(const int* p) { return USE_L1 ? __ldca(p) : __ldcg(p); }

template <bool USE_L1>
__global__ void __cluster_dims__(RV_CLUSTER, 1, 1) __launch_bounds__(RV_THREADS)
k_region_voting_global(AdcParams P, const uchar4* __restrict__ arms, float* disp_old, float* disp_new,
                       uint8_t* label, int* pend, int* counters, int* tile_stamp, int* last_eval) {
    extern __shared__ int rv_hist[];   // [RV_WARPS][D]: one histogram per warp (dynamic: up to 64 KB at D = 512)
    __shared__ int s_tot[RV_WARPS];
    const AdcDims& dm = P.dm;
    const int pair = blockIdx.x / RV_CLUSTER;
    const int crank = blockIdx.x % RV_CLUSTER;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int gwarp = crank * RV_WARPS + wid, n_gwarps = RV_CLUSTER * RV_WARPS;
    const int gtid = crank * RV_THREADS + tid, n_gthreads = RV_CLUSTER * RV_THREADS;
    const int W = dm.W, D = dm.D;
    const int tw = (W + RV_TILE - 1) / RV_TILE, th = (dm.H + RV_TILE - 1) / RV_TILE;
    const int reach = max(P.L1, 0);
    const uchar4* A = arms + (size_t)pair * dm.N;
    float* d_old = disp_old + (size_t)pair * dm.N;
    float* d_new = disp_new + (size_t)pair * dm.N;
    uint8_t* lab = label + (size_t)pair * dm.N;
    int* tiles = tile_stamp + (size_t)pair * tw * th;
    int* evalep = last_eval + (size_t)pair * dm.N;
    int* cnt = counters + pair * ADC_CNT;   // 0,1: list sizes   2: rounds   3: evaluations   4..6: change flags (mod 3)
    int n_list[2] = {__ldcg(cnt + 0), __ldcg(cnt + 1)};
    int rounds_total = 0, evals = 0;
    int* hist = rv_hist + wid * D;

    // nothing stamped, nothing evaluated: stamp(0) >= last_eval(0) makes the first round evaluate everyone
    for (int i = gtid; i < tw * th; i += n_gthreads) __stcg(tiles + i, 0);
    for (int k = 0; k < 2; k++) {
        const int* list = pend + ((size_t)pair * 2 + k) * dm.N;
        for (int i = gtid; i < n_list[k]; i += n_gthreads) __stcg(evalep + list[i], 0);
    }
    if (gtid < 3) __stcg(cnt + 4 + gtid, 0);
    int epoch = 1, rnd = 0;   // rnd indexes the three rotating change flags
    cluster_sync_all();

    for (int it = 0; it < 5; it++) {
        for (int k = 0; k < 2; k++) {
            int* list = pend + ((size_t)pair * 2 + k) * dm.N;
            const int n = n_list[k];
            if (n == 0) continue;  // uniform across the cluster
            bool any_fill = false;
            while (true) {
                if (gtid == 0) __stcg(cnt + 4 + (rnd + 1) % 3, 0);  // flag of the NEXT round; nobody reads it now
                bool warp_changed = false;
                for (int idx = gwarp; idx < n; idx += n_gwarps) {
                    const int p = rv_ld<USE_L1>(list + idx);
                    const int y = p / W, x = p - y * W;
                    if (rv_ld<USE_L1>(tiles + (y / RV_TILE) * tw + x / RV_TILE) < rv_ld<USE_L1>(evalep + p)) continue;  // inputs untouched since
                    evals++;
                    for (int b = lane; b < D; b += 32) hist[b] = 0;
                    __syncwarp();
                    const uchar4 a = __ldg(A + p);
                    // one region row per lane: the arm loads of all rows go out together, then every lane
                    // streams its own row segment (independent loads, several in flight)
                    for (int t = -(int)a.z + lane; t <= (int)a.w; t += 32) {
                        const int rowi = (y + t) * W + x;
                        const uchar4 a2 = __ldg(A + rowi);
                        const int s_lo = -(int)a2.x, s_hi = (int)a2.y;
                        const int s_mid = t < 0 ? s_hi + 1 : (t == 0 ? 0 : s_lo);   // first s that reads OLD
#pragma unroll 4
                        for (int s = s_lo; s <= s_hi; s++) {
                            const float d = s < s_mid ? rv_ld<USE_L1>(d_new + rowi + s) : rv_ld<USE_L1>(d_old + rowi + s);
                            if (d != ADC_INVALID_F) {
                                const int di = (int)roundf(d) - dm.dmin;  // lround: half away from zero
                                if (di >= 0 && di < D) atomicAdd(&hist[di], 1);
                            }
                        }
                    }
                    __syncwarp();
                    int peak = 0, best = 0x7fffffff, total = 0;
                    for (int b = lane; b < D; b += 32) {
                        const int h = hist[b];
                        if (peak < h) { peak = h; best = b; }
                        total += h;
                    }
                    const int gpeak = __reduce_max_sync(0xffffffffu, peak);
                    const int gbest = __reduce_min_sync(0xffffffffu, peak == gpeak ? best : 0x7fffffff);
                    total = __reduce_add_sync(0xffffffffu, total);
                    float r = ADC_INVALID_F;
                    if (gpeak > 0 && total > P.irv_ts &&
                        __fdiv_rn(__fmul_rn((float)gpeak, 1.0f), (float)total) > P.irv_th)
                        r = (float)(gbest + dm.dmin);
                    const bool changed = __float_as_uint(r) != __float_as_uint(__ldcg(d_new + p));
                    __syncwarp();
                    if (lane == 0) {
                        __stcg(evalep + p, epoch);
                        if (changed) __stcg(d_new + p, r);
                    }
                    if (changed) { rv_stamp_tiles(tiles, tw, th, x, y, reach, epoch, lane, 0); warp_changed = true; }
                }
                if (warp_changed && lane == 0) __stcg(cnt + 4 + rnd % 3, 1);
                cluster_sync_all();
                const int ch = __ldcg(cnt + 4 + rnd % 3);
                rounds_total++;
                epoch++;
                rnd++;
                if (!ch) break;
                any_fill = true;
            }
            if (!any_fill) continue;  // nothing was filled in this sweep: list and maps unchanged
            // ---- commit the sweep (OLD <- NEW for filled pixels; they become visible to everyone, so
            //      their neighbourhoods are stamped again), then erase them from the list
            for (int idx = gwarp; idx < n; idx += n_gwarps) {
                const int p = __ldcg(list + idx);
                const float v = __ldcg(d_new + p);
                if (v != ADC_INVALID_F) {
                    if (lane == 0) { __stcg(d_old + p, v); lab[p] = 0; }
                    const int y = p / W;
                    rv_stamp_tiles(tiles, tw, th, p - y * W, y, reach, epoch, lane, reach);
                }
            }
            epoch++;
            cluster_sync_all();
            if (crank == 0) {
                const int kept = rv_compact_invalid(n, list, d_old, s_tot);
                if (tid == 0) __stcg(cnt + k, kept);
            }
            cluster_sync_all();
            n_list[k] = __ldcg(cnt + k);
        }
    }
    evals = __reduce_add_sync(0xffffffffu, lane == 0 ? evals : 0);
    if (lane == 0) atomicAdd(cnt + 3, evals);
    if (gtid == 0) __stcg(cnt + 2, rounds_total);
}

// ---------------------------------------------------------------------------------------------
// Byte state for the fast voting kernel: only the rounded disparity index matters for a vote, so the
// state is one byte per pixel (0..253 = index, 254 = valid but outside [0,D), 255 = invalid).
// ---------------------------------------------------------------------------------------------
__global__ void k_vote_encode(AdcDims dm, const float* __restrict__ disp, const uchar4* __restrict__ arms,
                              uint8_t* __restrict__ dq, uchar2* __restrict__ alr, int* __restrict__ vstate) {   // dq: [2i] = NEW, [2i+1] = OLD
    const int pair = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= dm.N) return;
    const float d = disp[(size_t)pair * dm.N + i];
    uint8_t v = 255;
    if (d != ADC_INVALID_F) {
        const int di = (int)roundf(d) - dm.dmin;
        v = (di >= 0 && di < dm.D && di < 254) ? (uint8_t)di : (uint8_t)254;
    }
    reinterpret_cast<uchar2*>(dq + (size_t)pair * 2 * dm.N)[i] = make_uchar2(v, v);
    if (vstate) vstate[(size_t)pair * dm.N + i] = v == 255 ? -1 : (int)v;   // k_vote.cu: index of a valid pixel, -1 = invalid
    const uchar4 a = arms[(size_t)pair * dm.N + i];
    alr[(size_t)pair * dm.N + i] = make_uchar2(a.x, a.y);   // horizontal arms, 2 bytes per pixel
}

// ---------------------------------------------------------------------------------------------
// Byte-state version of the balanced cluster kernel (default).  Same algorithm as
// k_region_voting_global with two changes that matter for speed: (1) the per-round "does this pending
// pixel need another look?" test is done 32 list entries at a time, one per lane, instead of one
// dependent L2 round trip after the other per warp (that serial test loop, not the votes, dominated
// the first versions); (2) the state is one byte per pixel and the horizontal arms two, so a vote
// moves 4x fewer bytes.  Mutable state is read at L2 (ld.cg) -- the CTAs of the cluster sit on
// different SMs -- the constant arms through the read-only path.
// ---------------------------------------------------------------------------------------------
// (capping this kernel at 32 registers so that other lanes' kernels fit beside it was measured: slower overall)
__global__ void __cluster_dims__(RV_CLUSTER, 1, 1) __launch_bounds__(RV_THREADS)
k_region_voting_bytes(AdcParams P, const uchar4* __restrict__ arms, const uchar2* __restrict__ alr_all,
                      float* disp_old, float* disp_new, uint8_t* dq, uint8_t* label, int* pend, int* counters,
                      int* tile_stamp, int* last_eval) {
    __shared__ int s_hist[RV_WARPS][RV_MAXD];
    __shared__ int s_tot[RV_WARPS];
    const AdcDims& dm = P.dm;
    const int pair = blockIdx.x / RV_CLUSTER;
    const int crank = blockIdx.x % RV_CLUSTER;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int gwarp = crank * RV_WARPS + wid, n_gwarps = RV_CLUSTER * RV_WARPS;
    const int gtid = crank * RV_THREADS + tid, n_gthreads = RV_CLUSTER * RV_THREADS;
    const int W = dm.W, D = dm.D;
    const int tw = (W + RV_TILE - 1) / RV_TILE, th = (dm.H + RV_TILE - 1) / RV_TILE;
    const int reach = max(P.L1, 0);
    const uchar4* A = arms + (size_t)pair * dm.N;
    const uchar2* ALR = alr_all + (size_t)pair * dm.N;
    float* d_old = disp_old + (size_t)pair * dm.N;
    float* d_new = disp_new + (size_t)pair * dm.N;
    uint8_t* q2 = dq + (size_t)pair * 2 * dm.N;        // per pixel two bytes: [2p] = NEW state, [2p+1] = OLD state
    const unsigned short* q2w = reinterpret_cast<const unsigned short*>(q2);
    uint8_t* lab = label + (size_t)pair * dm.N;
    int* tiles = tile_stamp + (size_t)pair * tw * th;
    int* evalep = last_eval + (size_t)pair * dm.N;
    int* cnt = counters + pair * ADC_CNT;
    int n_list[2] = {__ldcg(cnt + 10), __ldcg(cnt + 11)};   // active (fillable) lists, see launch_active_lists
    int rounds_total = 0, evals = 0;
    int* hist = s_hist[wid];
    unsigned long long t_work = 0, t_bar = 0, t_commit = 0, t_compact = 0, t0 = 0;
    auto now = []() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; };

    for (int i = gtid; i < tw * th; i += n_gthreads) __stcg(tiles + i, 0);
    for (int k = 0; k < 2; k++) {
        const int* list = pend + ((size_t)pair * 2 + k) * dm.N;
        for (int i = gtid; i < n_list[k]; i += n_gthreads) __stcg(evalep + list[i], 0);
    }
    if (gtid < 3) __stcg(cnt + 4 + gtid, 0);
    int epoch = 1, rnd = 0;
    cluster_sync_all();

    for (int it = 0; it < 5; it++) {
        for (int k = 0; k < 2; k++) {
            int* list = pend + ((size_t)pair * 2 + k) * dm.N;
            const int n = n_list[k];
            if (n == 0) continue;  // uniform across the cluster
            bool any_fill = false;
            while (true) {
                if (gtid == 0) __stcg(cnt + 4 + (rnd + 1) % 3, 0);
                bool warp_changed = false;
                t0 = now();
                // 32 list entries per warp trip: every lane checks one pending pixel (is its tile stamped since
                // its last evaluation?), then the warp evaluates the dirty ones one after the other
                // (entries are dealt so that neighbouring list entries -- neighbouring pixels, which tend to be
                //  dirty together -- go to different warps: entry = trip*32*n_gwarps + lane*n_gwarps + gwarp)
                for (int base = 0; base < n; base += n_gwarps * 32) {
                    const int my = base + lane * n_gwarps + gwarp;
                    int p_l = 0;
                    unsigned tb_l = 0;
                    bool dirty_l = false;
                    if (my < n) {
                        p_l = __ldcg(list + my);
                        const int yy = p_l / W, xx = p_l - yy * W;
                        const uchar4 a_l = __ldg(A + p_l);
                        tb_l = (unsigned)a_l.z | ((unsigned)a_l.w << 8);
                        dirty_l = __ldcg(tiles + (yy / RV_TILE) * tw + xx / RV_TILE) >= __ldcg(evalep + p_l);
                    }
                    unsigned todo = __ballot_sync(0xffffffffu, dirty_l);
                    while (todo) {
                        const int src = __ffs(todo) - 1;
                        todo &= todo - 1;
                        const int p = __shfl_sync(0xffffffffu, p_l, src);
                        const unsigned tb = __shfl_sync(0xffffffffu, tb_l, src);
                        const int y = p / W, x = p - y * W;
                        evals++;
                        for (int b = lane; b < D; b += 32) hist[b] = 0;
                        __syncwarp();
                        // Region scan.  The horizontal arms of all (<= 69) region rows are fetched in ONE round of loads
                        // (three per lane at most) and handed out by shuffle; then the region is visited in trips of
                        // 4 rows x 16 columns, software-pipelined (the loads of trip j+1 are in flight while trip j is
                        // added to the histogram).  Trip count = ceil(rows/4) x ceil(longest row/16): small regions cost
                        // few instructions.  One 16-bit load brings a pixel's NEW and OLD state; it goes through L1
                        // (ld.ca): neighbouring pixels are evaluated on the same SM and share their regions, and every
                        // cluster barrier ends in CCTL.IVALL (see the SASS), so no line outlives a round.  A line going
                        // stale inside a round is harmless (asynchronous fixed point; the certifying round writes nothing).
                        const int top = (int)(tb & 255u), rows = top + (int)(tb >> 8) + 1;
                        const int rbase = (y - top) * W + x;
                        unsigned ar0, ar1 = 0, ar2 = 0;
                        {
                            const uchar2 v = lane < rows ? __ldg(ALR + rbase + lane * W) : make_uchar2(0, 0);
                            ar0 = (unsigned)v.x | ((unsigned)v.y << 8);
                        }
                        if (rows > 32) {
                            const uchar2 v1 = lane + 32 < rows ? __ldg(ALR + rbase + (lane + 32) * W) : make_uchar2(0, 0);
                            const uchar2 v2 = lane + 64 < rows ? __ldg(ALR + rbase + (lane + 64) * W) : make_uchar2(0, 0);
                            ar1 = (unsigned)v1.x | ((unsigned)v1.y << 8);
                            ar2 = (unsigned)v2.x | ((unsigned)v2.y << 8);
                        }
                        const int span_l = (int)(ar0 & 255u) + (int)(ar0 >> 8);
                        const int span_m = max(span_l, max((int)(ar1 & 255u) + (int)(ar1 >> 8), (int)(ar2 & 255u) + (int)(ar2 >> 8)));
                        const int ncp = (__reduce_max_sync(0xffffffffu, span_m) >> 4) + 1;   // 16-column chunks per row
                        const int grp = lane >> 3, sub = lane & 7;
                        const int n_trips = ((rows + 3) >> 2) * ncp;
                        int ti = 0, tc = 0;                        // row group / column chunk of the trip being FETCHED
                        auto fetch_trip = [&](int& o0, int& o1) {
                            const int ri = 4 * ti + grp;
                            unsigned a2 = __shfl_sync(0xffffffffu, ar0, ri & 31);
                            if (rows > 32) {
                                const unsigned a2b = __shfl_sync(0xffffffffu, ar1, ri & 31);
                                const unsigned a2c = __shfl_sync(0xffffffffu, ar2, ri & 31);
                                a2 = ri < 32 ? a2 : (ri < 64 ? a2b : a2c);
                            }
                            const int s_hi = ri < rows ? (int)(a2 >> 8) : -0x10000;       // dead rows: empty segment
                            const int s0 = -(int)(a2 & 255u) + sub + 16 * tc, s1 = s0 + 8;
                            const int t = ri - top;
                            const int mid = t < 0 ? 0x10000 : (t == 0 ? 0 : -0x10000);   // columns below `mid` read NEW
                            const unsigned short* rp = q2w + rbase + ri * W;
                            o0 = o1 = 255;
                            if (s0 <= s_hi) { const unsigned w2 = __ldca(rp + s0); o0 = s0 < mid ? (int)(w2 & 255u) : (int)(w2 >> 8); }
                            if (s1 <= s_hi) { const unsigned w2 = __ldca(rp + s1); o1 = s1 < mid ? (int)(w2 & 255u) : (int)(w2 >> 8); }
                            if (++tc == ncp) { tc = 0; ti++; }
                        };
                        int d0, d1;
                        fetch_trip(d0, d1);
                        for (int j = 0; j < n_trips; j++) {
                            int n0 = 255, n1 = 255;
                            if (j + 1 < n_trips) fetch_trip(n0, n1);
                            if (d0 < 254) atomicAdd(&hist[d0], 1);
                            if (d1 < 254) atomicAdd(&hist[d1], 1);
                            d0 = n0; d1 = n1;
                        }
                        __syncwarp();
                        int peak = 0, best = 0x7fffffff, total = 0;
                        for (int b = lane; b < D; b += 32) {
                            const int h = hist[b];
                            if (peak < h) { peak = h; best = b; }
                            total += h;
                        }
                        const int gpeak = __reduce_max_sync(0xffffffffu, peak);
                        const int gbest = __reduce_min_sync(0xffffffffu, peak == gpeak ? best : 0x7fffffff);
                        total = __reduce_add_sync(0xffffffffu, total);
                        int r = 255;
                        if (gpeak > 0 && total > P.irv_ts &&
                            __fdiv_rn(__fmul_rn((float)gpeak, 1.0f), (float)total) > P.irv_th)
                            r = gbest;
                        const bool changed = r != (int)__ldcg(q2 + 2 * p);
                        __syncwarp();
                        if (lane == 0) {
                            __stcg(evalep + p, epoch);
                            if (changed) __stcg(q2 + 2 * p, (uint8_t)r);
                        }
                        if (changed) { rv_stamp_tiles(tiles, tw, th, x, y, reach, epoch, lane, 0); warp_changed = true; }
                    }
                }
                if (warp_changed && lane == 0) __stcg(cnt + 4 + rnd % 3, 1);
                { const unsigned long long t1 = now(); t_work += t1 - t0; t0 = t1; }
                cluster_sync_all();
                { const unsigned long long t1 = now(); t_bar += t1 - t0; t0 = t1; }
                const int ch = __ldcg(cnt + 4 + rnd % 3);
                rounds_total++;
                epoch++;
                rnd++;
                if (!ch) break;
                any_fill = true;
            }
            if (!any_fill) continue;
            t0 = now();
            for (int base = gwarp * 32; base < n; base += n_gwarps * 32) {   // one list entry per lane
                const int my = base + lane;
                int p_l = 0, v_l = 255;
                if (my < n) { p_l = __ldcg(list + my); v_l = __ldcg(q2 + 2 * p_l); }
                if (v_l != 255) {
                    const float f = (float)(v_l + dm.dmin);
                    __stcg(q2 + 2 * p_l + 1, (uint8_t)v_l);
                    __stcg(d_old + p_l, f);
                    __stcg(d_new + p_l, f);
                    __stcg(lab + p_l, (uint8_t)0);
                }
                unsigned filled = __ballot_sync(0xffffffffu, v_l != 255);
                while (filled) {
                    const int src = __ffs(filled) - 1;
                    filled &= filled - 1;
                    const int p = __shfl_sync(0xffffffffu, p_l, src);
                    const int y = p / W;
                    rv_stamp_tiles(tiles, tw, th, p - y * W, y, reach, epoch, lane, reach);
                }
            }
            epoch++;
            cluster_sync_all();
            { const unsigned long long t1 = now(); t_commit += t1 - t0; t0 = t1; }
            if (crank == 0) {
                const int kept = rv_compact_invalid(n, list, d_old, s_tot);
                if (tid == 0) __stcg(cnt + 10 + k, kept);
            }
            cluster_sync_all();
            { const unsigned long long t1 = now(); t_compact += t1 - t0; t0 = t1; }
            n_list[k] = __ldcg(cnt + 10 + k);
        }
    }
    evals = __reduce_add_sync(0xffffffffu, lane == 0 ? evals : 0);
    if (lane == 0) atomicAdd(cnt + 3, evals);
    if (gtid == 0) {
        __stcg(cnt + 2, rounds_total);
        __stcg(cnt + 12, (int)(t_work / 1000)); __stcg(cnt + 13, (int)(t_bar / 1000));     // warp 0's view, microseconds
        __stcg(cnt + 14, (int)(t_commit / 1000)); __stcg(cnt + 15, (int)(t_compact / 1000));
    }
}

// Three kernels, chosen by the parameters alone (each has its parity cases in tests/test_gpu_parity.py):
//   D <= 254 and L1 <= 127   incremental histograms, k_vote.cu (every BASELINE configuration)
//   D <= 254, L1 > 127       byte-state pull kernel (a cross region may hold more than 65535 pixels)
//   D = 255 .. 512           float-state pull kernel (the byte state codes a disparity index in one byte)
#define RV_GLOBAL_SMEM_ATTR (RV_WARPS * 512 * 4)
size_t adc_voting_smem(const AdcDims& dm, size_t* cap) {
    *cap = RV_GLOBAL_SMEM_ATTR;
    return dm.D <= 254 ? 0 : (size_t)RV_WARPS * dm.D * 4;   // (the D <= 254 kernels' histograms are static / budgeted in k_vote.cu)
}

void adc_launch_voting(const AdcParams& P, const AdcWave& w, cudaStream_t st, unsigned long long* launches) {
    // disp_l = committed state (OLD), disp_t = working copy (NEW); both hold the post-outlier map here
    dim3 egrid((P.dm.N + 255) / 256, w.S);
    if (P.dm.D <= 254) {
        launch_active_lists(P, w, st, launches);
        k_vote_encode<<<egrid, 256, 0, st>>>(P.dm, w.disp_l, w.arms, w.vote_dq, w.vote_alr, w.vote_state);
        ++*launches;
        if (!adc_launch_vote_push(P, w, st, launches)) {
            k_region_voting_bytes<<<w.S * RV_CLUSTER, RV_THREADS, 0, st>>>(P, w.arms, w.vote_alr, w.disp_l, w.disp_t, w.vote_dq,
                                                                          w.label, w.vlist, w.counters, w.tile_stamp, w.last_eval);
            ++*launches;
        }
        adc_launch_build_lists(P, w, st, launches);   // outlier lists = every listed pixel that is still invalid
    } else {
        static AdcOnce attr_once;
        if (adc_once_needed(attr_once)) {
            cudaFuncSetAttribute(k_region_voting_global<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, RV_GLOBAL_SMEM_ATTR);
            adc_once_done(attr_once);
        }
        size_t cap;
        k_region_voting_global<false><<<w.S * RV_CLUSTER, RV_THREADS, adc_voting_smem(P.dm, &cap), st>>>(
            P, w.arms, w.disp_l, w.disp_t, w.label, w.pend, w.counters, w.tile_stamp, w.last_eval);
        ++*launches;
    }
}

// =============================================================================================
// 3. Proper interpolation.  For each pixel still in a list: 16 rays (angle accumulated in double
//    from the float quotient 3.1415926f/16), first valid disparity met along each; mismatches take
//    the candidate whose colour is closest (first wins), occlusions the smallest disparity; no
//    candidate -> 0.0 (the reference's value-initialised fill vector).  Results of one list are
//    written after the whole list has been evaluated (Jacobi), the occlusion list then sees the
//    filled mismatches -- hence one launch per list reading disp_old and writing disp_new.
//    The ray coordinates are evaluated exactly as the reference does, lround(y + m*sin) in double
//    without contraction, with sin/cos tables from the host's libm.
//    16 lanes = 16 rays of one pixel; two pixels per warp.
// =============================================================================================
__global__ void __launch_bounds__(256)
k_interpolate(AdcParams P, int k, const uint8_t* __restrict__ bgr, const float* __restrict__ disp_old,
              float* __restrict__ disp_new, const int* __restrict__ pend, const int* __restrict__ counters,
              const double* __restrict__ ray_sin, const double* __restrict__ ray_cos,
              const short2* __restrict__ ray_off) {
    const AdcDims& dm = P.dm;
    const int pair = blockIdx.y;
    const int n = counters[pair * ADC_CNT + k];
    const int* list = pend + ((size_t)pair * 2 + k) * dm.N;
    const uint8_t* left = bgr + (size_t)pair * 2 * dm.N * 3;
    const float* d_old = disp_old + (size_t)pair * dm.N;
    float* d_new = disp_new + (size_t)pair * dm.N;
    const int ray = threadIdx.x & 15;
    const int slot = (blockIdx.x * blockDim.x + threadIdx.x) >> 4;
    const int n_slots = (gridDim.x * blockDim.x) >> 4;
    const unsigned half_mask = 0xffffu << (threadIdx.x & 16);
    const double sa = ray_sin[ray], ca = ray_cos[ray];
    for (int base = 0; base < n; base += n_slots) {   // uniform trip count for the whole warp
        const int idx = base + slot;
        const bool active = idx < n;
        int p = 0, x = 0, y = 0;
        if (active) { p = list[idx]; y = p / dm.W; x = p - y * dm.W; }
        int dist = 0x7fffffff;
        float dval = ADC_LARGE_F;
        bool found = false;
        if (active) {
            const uchar3 c0 = adc_load_bgr(left, p);
            for (int m = 1; m < P.max_search; m++) {
                long yy, xx;
                if (ray_off) {   // integer offsets, verified on the host to equal the expression below for this image size
                    const short2 o = __ldg(ray_off + ray * P.max_search + m);
                    yy = y + o.y; xx = x + o.x;
                } else {
                    yy = lround(__dadd_rn((double)y, __dmul_rn((double)m, sa)));
                    xx = lround(__dadd_rn((double)x, __dmul_rn((double)m, ca)));
                }
                if (yy < 0 || yy >= dm.H || xx < 0 || xx >= dm.W) break;
                const int q = (int)yy * dm.W + (int)xx;
                const float d = d_old[q];
                if (d != ADC_INVALID_F) {
                    const uchar3 c = adc_load_bgr(left, q);
                    dist = abs((int)c0.x - (int)c.x) + abs((int)c0.y - (int)c.y) + abs((int)c0.z - (int)c.z);
                    dval = d;
                    found = true;
                    break;
                }
            }
        }
        // combine the 16 rays of this pixel (half-warp)
        const unsigned any = __ballot_sync(0xffffffffu, found) & half_mask;
        float result = 0.0f;
        if (k == 0) {
            // smallest colour distance, earliest ray on ties (strict '>' in the reference, min_dist starts at 9999)
            int key = (found && dist < 9999) ? ((dist << 4) | ray) : 0x7fffffff;
#pragma unroll
            for (int o = 8; o >= 1; o >>= 1) key = min(key, __shfl_xor_sync(0xffffffffu, key, o));
            const int win = key & 15;
            const float dw = __shfl_sync(0xffffffffu, dval, (threadIdx.x & 16) | win);
            if (key != 0x7fffffff) result = dw;     // all candidates farther than 9999 keep d = 0.0f
        } else {
            float mv = found ? dval : ADC_LARGE_F;
#pragma unroll
            for (int o = 8; o >= 1; o >>= 1) mv = fminf(mv, __shfl_xor_sync(0xffffffffu, mv, o));
            result = mv;
        }
        if (any == 0) result = 0.0f;
        if (active && ray == 0) d_new[p] = result;
    }
}

// Fast path of the same step, used when the integer ray table is available (it is whenever it was verified exact
// for this image size, see engine.cu).  The generic kernel spends ~15 instructions per ray step on coordinates,
// four bounds tests and a float load; here the walk runs on a padded byte map (0 = invalid pixel: keep going,
// 1 = valid: candidate found, 2 = outside the image: the ray ends) with the ray table in shared memory as linear
// offsets into that map: one shared load, one add, one byte load and a test per step.
__global__ void __launch_bounds__(256)
k_interp_map(AdcDims dm, int B, const float* __restrict__ disp, uint8_t* __restrict__ imap) {
    const int Wp = dm.W + 2 * B, Hp = dm.H + 2 * B;
    const int pair = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Wp * Hp) return;
    const int yp = i / Wp, xp = i - yp * Wp;
    const int y = yp - B, x = xp - B;
    uint8_t v = 2;
    if (y >= 0 && y < dm.H && x >= 0 && x < dm.W) v = disp[(size_t)pair * dm.N + y * dm.W + x] != ADC_INVALID_F ? 1 : 0;
    imap[(size_t)pair * Wp * Hp + i] = v;
}

__global__ void __launch_bounds__(256)
k_interpolate_fast(AdcParams P, int k, const unsigned* __restrict__ bgrx, const float* __restrict__ disp_old,
                   float* __restrict__ disp_new, const int* __restrict__ pend, const int* __restrict__ counters,
                   const short2* __restrict__ ray_off, const uint8_t* __restrict__ imap_all) {
    extern __shared__ int ip_off[];   // [16][max_search]: dy * Wp + dx
    const AdcDims& dm = P.dm;
    const int L = P.max_search, B = L - 1, Wp = dm.W + 2 * B, Hp = dm.H + 2 * B;
    for (int i = threadIdx.x; i < 16 * L; i += blockDim.x) { const short2 o = ray_off[i]; ip_off[i] = (int)o.y * Wp + (int)o.x; }
    __syncthreads();
    const int pair = blockIdx.y;
    const int n = counters[pair * ADC_CNT + k];
    const int* list = pend + ((size_t)pair * 2 + k) * dm.N;
    const unsigned* left = bgrx + (size_t)pair * 2 * dm.N;   // packed B | G<<8 | R<<16
    const float* d_old = disp_old + (size_t)pair * dm.N;
    float* d_new = disp_new + (size_t)pair * dm.N;
    const uint8_t* imap = imap_all + (size_t)pair * Wp * Hp;
    const int ray = threadIdx.x & 15;
    const int slot = (blockIdx.x * blockDim.x + threadIdx.x) >> 4;
    const int n_slots = (gridDim.x * blockDim.x) >> 4;
    const unsigned half_mask = 0xffffu << (threadIdx.x & 16);
    const int* myoff = ip_off + ray * L;
    for (int base = 0; base < n; base += n_slots) {   // uniform trip count for the whole warp
        const int idx = base + slot;
        const bool active = idx < n;
        int p = 0;
        int dist = 0x7fffffff;
        float dval = ADC_LARGE_F;
        bool found = false;
        if (active) {
            p = list[idx];
            const int y = p / dm.W, x = p - y * dm.W;
            const uint8_t* c0p = imap + (y + B) * Wp + (x + B);
            int m = 1, hit = 2;
            for (; m < L; m++) {
                hit = c0p[myoff[m]];
                if (hit) break;
            }
            if (m < L && hit == 1) {
                const short2 o = __ldg(ray_off + ray * L + m);
                const int q = (y + o.y) * dm.W + (x + o.x);
                const unsigned a = __ldg(left + p), b = __ldg(left + q);
                const unsigned ad = __vabsdiffu4(a, b);
                dist = (int)(ad & 255u) + (int)((ad >> 8) & 255u) + (int)((ad >> 16) & 255u);
                dval = d_old[q];
                found = true;
            }
        }
        // combine the 16 rays of this pixel (half-warp) -- as in k_interpolate
        const unsigned any = __ballot_sync(0xffffffffu, found) & half_mask;
        float result = 0.0f;
        if (k == 0) {
            int key = (found && dist < 9999) ? ((dist << 4) | ray) : 0x7fffffff;
#pragma unroll
            for (int o = 8; o >= 1; o >>= 1) key = min(key, __shfl_xor_sync(0xffffffffu, key, o));
            const int win = key & 15;
            const float dw = __shfl_sync(0xffffffffu, dval, (threadIdx.x & 16) | win);
            if (key != 0x7fffffff) result = dw;
        } else {
            float mv = found ? dval : ADC_LARGE_F;
#pragma unroll
            for (int o = 8; o >= 1; o >>= 1) mv = fminf(mv, __shfl_xor_sync(0xffffffffu, mv, o));
            result = mv;
        }
        if (any == 0) result = 0.0f;
        if (active && ray == 0) d_new[p] = result;
    }
}

void adc_launch_interp_list(const AdcParams& P, const AdcWave& w, int k, cudaStream_t st, unsigned long long* launches) {
    dim3 grid(592, w.S);
    const int L = P.max_search, B = L - 1;
    const size_t map_bytes = (size_t)(P.dm.W + 2 * B) * (P.dm.H + 2 * B);
    if (w.ray_off && L >= 2 && map_bytes <= (size_t)P.dm.N * 8 && (size_t)16 * L * sizeof(int) <= 48 * 1024) {
        uint8_t* imap = reinterpret_cast<uint8_t*>(w.vote_dirty);   // [S][N] int2 scratch of the voting step, idle by now
        dim3 mgrid((unsigned)((map_bytes + 255) / 256), w.S);
        k_interp_map<<<mgrid, 256, 0, st>>>(P.dm, B, w.disp_l, imap);
        k_interpolate_fast<<<grid, 256, (size_t)16 * L * sizeof(int), st>>>(P, k, w.bgrx, w.disp_l, w.disp_t, w.pend, w.counters,
                                                                            w.ray_off, imap);
        *launches += 2;
        return;
    }
    k_interpolate<<<grid, 256, 0, st>>>(P, k, w.bgr, w.disp_l, w.disp_t, w.pend, w.counters, w.ray_sin, w.ray_cos, w.ray_off);
    ++*launches;
}

// Origin map (side output, adcensus_b200.h ADC_ORIGIN_*), after the last filling step that ran.  Every voting kernel
// clears the label of a pixel it fills and interpolation leaves the labels alone, so: a pixel listed before voting
// (lab0) and no longer listed after it was filled by voting; one still listed and now finite, by interpolation.  Without
// filling the labels never change, and every listed pixel is still Invalid_Float.  origin holds the WTA-invalid flag.
__global__ void k_origin(AdcDims dm, const uint8_t* __restrict__ lab0, const uint8_t* __restrict__ lab1,
                         const float* __restrict__ disp, uint8_t* __restrict__ origin) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= dm.N) return;
    const size_t o = (size_t)blockIdx.y * dm.N + i;
    const uint8_t l0 = lab0[o];
    uint8_t code = ADC_ORIGIN_MATCHED;
    if (disp[o] == ADC_INVALID_F) code = ADC_ORIGIN_INVALID;
    else if (l0 != 0) code = lab1[o] == 0 ? l0 : (uint8_t)(l0 + 2);   // 1, 2: voted mismatch / occlusion; 3, 4: interpolated
    origin[o] |= code;
}

void adc_launch_origin(const AdcParams& P, const AdcWave& w, const AdcAux& aux, cudaStream_t st, unsigned long long* launches) {
    dim3 grid((P.dm.N + 255) / 256, w.S);
    k_origin<<<grid, 256, 0, st>>>(P.dm, aux.lab0, w.label, w.disp_l, aux.origin);
    ++*launches;
}

// =============================================================================================
// 4. Depth-discontinuity adjustment (default OFF in ADCensusOption).  Sobel edge mask on the
//    disparity map, then per row a strictly sequential left-to-right pass (pixel x may copy from
//    x-1, which may itself have just been changed) -> one thread per row.  The reference indexes
//    the cost volume with lround(d) without subtracting dmin (multistep_refiner.cpp:331); indices
//    outside [0,D) are undefined behaviour there and skipped here (the CPU checker does the same).
// =============================================================================================
__global__ void k_edge_mask(AdcDims dm, const float* __restrict__ disp, uint8_t* __restrict__ edge) {
    const int pair = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= dm.N) return;
    const int y = i / dm.W, x = i - y * dm.W;
    uint8_t e = 0;
    if (y >= 1 && y < dm.H - 1 && x >= 1 && x < dm.W - 1) {
        const float* r1 = disp + (size_t)pair * dm.N + i;
        const float* r0 = r1 - dm.W;
        const float* r2 = r1 + dm.W;
        const float A = __fadd_rn(-r0[-1], r0[1]);
        const float B = __fadd_rn(__fmul_rn(-2.0f, r1[-1]), __fmul_rn(2.0f, r1[1]));
        const float C = __fadd_rn(-r2[-1], r2[1]);
        const float gx = __fadd_rn(__fadd_rn(A, B), C);
        const float T = __fsub_rn(__fsub_rn(-r0[-1], __fmul_rn(2.0f, r0[0])), r0[1]);
        const float U = __fadd_rn(__fadd_rn(r2[-1], __fmul_rn(2.0f, r2[0])), r2[1]);
        const float gy = __fadd_rn(T, U);
        if (__fadd_rn(fabsf(gx), fabsf(gy)) > 5.0f) e = 1;
    }
    edge[(size_t)pair * dm.N + i] = e;
}

__global__ void k_discontinuity_rows(AdcDims dm, float* __restrict__ disp, const uint8_t* __restrict__ edge,
                                     const float* __restrict__ vol) {
    const int pair = blockIdx.y;
    const int y = blockIdx.x * blockDim.x + threadIdx.x;
    if (y >= dm.H) return;
    float* row = disp + (size_t)pair * dm.N + (size_t)y * dm.W;
    const uint8_t* erow = edge + (size_t)pair * dm.N + (size_t)y * dm.W;
    for (int x = 1; x < dm.W - 1; x++) {
        if (erow[x] != 1) continue;
        const float d = row[x];
        if (d == ADC_INVALID_F) continue;
        const float* cost = vol + (size_t)pair * dm.vol_stride + ((size_t)y * dm.W + x) * dm.Dp;
        const long di = lroundf(d);
        if (di < 0 || di >= dm.D) continue;
        float c0 = cost[di];
        for (int k = 0; k < 2; k++) {
            const float d2 = row[k == 0 ? x - 1 : x + 1];
            if (d2 == ADC_INVALID_F) continue;
            const long d2i = lroundf(d2);
            if (d2i < 0 || d2i >= dm.D) continue;
            const float cc = k == 0 ? cost[-dm.Dp + d2i] : cost[dm.Dp + d2i];
            if (cc < c0) { row[x] = d2; c0 = cc; }
        }
    }
}

void adc_launch_discontinuity(const AdcParams& P, const AdcWave& w, const float* vol, cudaStream_t st, unsigned long long* launches) {
    dim3 grid((P.dm.N + 255) / 256, w.S);
    k_edge_mask<<<grid, 256, 0, st>>>(P.dm, w.disp_l, w.flag);
    dim3 grid2((P.dm.H + 63) / 64, w.S);
    k_discontinuity_rows<<<grid2, 64, 0, st>>>(P.dm, w.disp_l, w.flag, vol);
    *launches += 2;
}

// =============================================================================================
// 5. In-place 3x3 median in raster order.  out(y,x) sees already-filtered values in row y-1 and
//    at (y,x-1), and original values elsewhere.  (y,x) depends on (y,x-1) and (y-1,x+1), so all
//    pixels with x + 2y = t are independent: a wavefront over t = 0 .. W+2H-3 with a CTA barrier
//    per step reproduces the sequential scan exactly (every window element of step t was produced
//    at a step != t).  Window = in-image neighbours, sorted, element n/2 (9->[4], 6->[3], 4->[2]);
//    realised as the median of 9 after padding with -inf/+inf so that the rank is preserved.
//    Data movement: one thread per row.  "Original" values come from the untouched input map
//    (read-only, so they cache in L1), "filtered" values of the row above come from a 4-deep
//    per-row ring in shared memory written by the neighbouring thread, the filtered left
//    neighbour is the thread's own previous result; the output goes to a second map.
// =============================================================================================
#define MED_THREADS 1024

__device__ __forceinline__ void cswap(float& a, float& b) { const float lo = fminf(a, b), hi = fmaxf(a, b); a = lo; b = hi; }

__device__ __forceinline__ float median9(float v[9]) {
    // 19-exchange median-of-9 selection network (Paeth / Smith)
    cswap(v[1], v[2]); cswap(v[4], v[5]); cswap(v[7], v[8]);
    cswap(v[0], v[1]); cswap(v[3], v[4]); cswap(v[6], v[7]);
    cswap(v[1], v[2]); cswap(v[4], v[5]); cswap(v[7], v[8]);
    cswap(v[0], v[3]); cswap(v[5], v[8]); cswap(v[4], v[7]);
    cswap(v[3], v[6]); cswap(v[1], v[4]); cswap(v[2], v[5]);
    cswap(v[4], v[7]); cswap(v[4], v[2]); cswap(v[6], v[4]);
    cswap(v[4], v[2]);
    return v[4];
}


__device__ __forceinline__ void med_cp4(float* smem_dst, const float* gmem_src) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(s), "l"(gmem_src) : "memory");
}

template <int MED_ROWS, int MED_PF>   // rows per thread (1 for H <= 1024, 2 up to 2048, 4 up to 4096); wavefront steps between issuing a load and using it
__global__ void __launch_bounds__(MED_THREADS)
k_median_wavefront(AdcDims dm, const float* __restrict__ in, float* __restrict__ out) {
    extern __shared__ float med_smem[];
    const int MT = blockDim.x;   // threads actually launched (rows rounded up to whole warps)
    // [H][4]: filtered values of each row, indexed by column & 3
    // then per thread and row: MED_PF slots x 2 floats of ORIGINAL values (row y, row y+1) of the column that
    // enters the window at a given step, filled by 4-byte cp.async issued MED_PF steps ahead
    const int pair = blockIdx.x;
    const float* src = in + (size_t)pair * dm.N;
    float* dst = out + (size_t)pair * dm.N;
    const int W = dm.W, H = dm.H;
    float* med_ring = med_smem;
    float* stage = med_smem + (size_t)H * 4 + (size_t)threadIdx.x * (MED_ROWS * MED_PF * 2);
    (void)MT;
    const float NINF = __int_as_float(0xff800000), PINF = ADC_INVALID_F;
    const int n_steps = W + 2 * H - 2;
    float A0[MED_ROWS], A1[MED_ROWS], Bm[MED_ROWS], B0[MED_ROWS], B1[MED_ROWS], left_new[MED_ROWS];
    auto issue = [&](int r, int t, int slot) {   // originals of column x + 1 = (t - 2y) + 1, consumed at step t
        const int y = threadIdx.x + r * MT;
        const int c = t - 2 * y + 1;
        float* s2 = stage + (r * MED_PF + slot) * 2;
        const bool ok = y < H && c >= 0 && c < W;
        if (ok) med_cp4(s2, src + y * W + c); else s2[0] = PINF;
        if (ok && y + 1 < H) med_cp4(s2 + 1, src + (y + 1) * W + c); else s2[1] = PINF;
    };
#pragma unroll
    for (int r = 0; r < MED_ROWS; r++) { A0[r] = A1[r] = Bm[r] = B0[r] = B1[r] = PINF; left_new[r] = PINF; }
#pragma unroll
    for (int j = 0; j < MED_PF; j++) {
#pragma unroll
        for (int r = 0; r < MED_ROWS; r++) issue(r, j - 2, j);
        asm volatile("cp.async.commit_group;\n" ::: "memory");
    }
    for (int tb = -2; tb < n_steps; tb += MED_PF) {
#pragma unroll
        for (int j = 0; j < MED_PF; j++) {
            const int t = tb + j;
            asm volatile("cp.async.wait_group %0;\n" ::"n"(MED_PF - 1) : "memory");   // this thread's copies for step t
            float res[MED_ROWS];
            bool act[MED_ROWS];
#pragma unroll
            for (int r = 0; r < MED_ROWS; r++) {
                const int y = threadIdx.x + r * MT;
                const int x = t - 2 * y;
                act[r] = false;
                res[r] = 0.f;
                if (x < -2 - MED_PF || x >= W) continue;   // this row's turn is far away or over: nothing to shift, fetch or compute
                const float* s2 = stage + (r * MED_PF + j) * 2;
                A0[r] = A1[r]; A1[r] = s2[0];
                Bm[r] = B0[r]; B0[r] = B1[r]; B1[r] = s2[1];
                issue(r, t + MED_PF, j);
                act[r] = t < n_steps && y < H && x >= 0 && x < W;
                if (!act[r]) continue;
                const bool up = y > 0, dn = y + 1 < H, lf = x > 0, rt = x + 1 < W;
                float v[9];
                const float* ring_up = med_ring + (size_t)(y - 1) * 4;
                v[0] = (up && lf) ? ring_up[(x - 1) & 3] : PINF;
                v[1] = up ? ring_up[x & 3] : PINF;
                v[2] = (up && rt) ? ring_up[(x + 1) & 3] : PINF;
                v[3] = lf ? left_new[r] : PINF;
                v[4] = A0[r];
                v[5] = rt ? A1[r] : PINF;
                v[6] = (dn && lf) ? Bm[r] : PINF;
                v[7] = dn ? B0[r] : PINF;
                v[8] = (dn && rt) ? B1[r] : PINF;
                const int n = (1 + (int)up + (int)dn) * (1 + (int)lf + (int)rt);
                int need = 4 - n / 2;   // rank n/2 of n values == rank 4 of 9 with (4 - n/2) absent slots at -inf
                const bool present[9] = {up && lf, up, up && rt, lf, true, rt, dn && lf, dn, dn && rt};
#pragma unroll
                for (int q = 0; q < 9; q++)
                    if (!present[q] && need > 0) { v[q] = NINF; need--; }
                res[r] = median9(v);
            }
            asm volatile("cp.async.commit_group;\n" ::: "memory");
            // Publish the results of this step.  Row y writes ring slot (x & 3); during this same step row y+1
            // (at column x-2) reads slots (x-3..x-1) & 3 of row y -- three slots that differ from x & 3 -- so the
            // writes need no barrier of their own; one barrier per step makes them visible to the next step.
#pragma unroll
            for (int r = 0; r < MED_ROWS; r++) {
                if (!act[r]) continue;
                const int y = threadIdx.x + r * MT;
                const int x = t - 2 * y;
                med_ring[(size_t)y * 4 + (x & 3)] = res[r];
                left_new[r] = res[r];
                dst[y * W + x] = res[r];
            }
            __syncthreads();
        }
    }
    asm volatile("cp.async.wait_group 0;\n" ::: "memory");
}

int adc_launch_median(const AdcParams& P, const AdcWave& w, const float* in, float* out, cudaStream_t st,
                      unsigned long long* launches) {
    if (P.dm.H > MED_THREADS * 4) return 1;        // (adc_create rejects such images: ADC_MAX_HEIGHT)
    const int rows = P.dm.H <= MED_THREADS ? 1 : (P.dm.H <= 2 * MED_THREADS ? 2 : 4);
    const int pf = rows == 4 ? 4 : 8;
    const int threads = std::min(MED_THREADS, ((P.dm.H + rows - 1) / rows + 31) / 32 * 32);
    const size_t smem = ((size_t)P.dm.H * 4 + (size_t)threads * rows * pf * 2) * sizeof(float);
    static AdcOnce attr_once;
    if (adc_once_needed(attr_once)) {
        cudaFuncSetAttribute(k_median_wavefront<1, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        cudaFuncSetAttribute(k_median_wavefront<2, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        cudaFuncSetAttribute(k_median_wavefront<4, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        adc_once_done(attr_once);
    }
    if (rows == 1)      k_median_wavefront<1, 8><<<w.S, threads, smem, st>>>(P.dm, in, out);
    else if (rows == 2) k_median_wavefront<2, 8><<<w.S, threads, smem, st>>>(P.dm, in, out);
    else                k_median_wavefront<4, 4><<<w.S, threads, smem, st>>>(P.dm, in, out);
    ++*launches;
    return 0;
}
