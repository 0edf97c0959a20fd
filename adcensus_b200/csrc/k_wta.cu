// k_wta.cu -- stage 4: winner-takes-all with parabola refinement for the left view and, from the
// same volume, for the right view (reference: ADCensusStereo.cpp:188-243 and :245-310).
#include "adc_common.cuh"
#include "../../include/adcensus_b200.h"

// Parabola through (best-1, best, best+1), ADCensusStereo.cpp:234-240.  Explicit _rn intrinsics keep
// nvcc from contracting c1 + c2 - 2*min into an FMA.
__device__ __forceinline__ float adc_subpixel(float c1, float c2, float cmin, int best) {
    const float denom = __fsub_rn(__fadd_rn(c1, c2), __fmul_rn(2.0f, cmin));
    if (denom != 0.0f) return __fadd_rn((float)best, __fdiv_rn(__fsub_rn(c1, c2), __fmul_rn(denom, 2.0f)));
    return (float)best;
}

// ---------------------------------------------------------------------------------------------
// One kernel, both views, any disparity range.  A CTA owns WT_PX neighbouring pixels of one image row -- as pixels of
// the left view AND as pixels of the right view -- and sweeps the disparity range in chunks of WT_DC.  Per chunk two
// small tiles are staged in shared memory (coalesced 128-bit loads, issued one chunk ahead: they land in registers while
// the previous chunk is scanned):
//   left tile   L[t][k] = cost(x0 + t, d0 + k)                          the chunk of the CTA's own columns
//   right tile  R[k][r] = cost(x0 + r + dmin + d0 + k, d0 + k)          cost_R(xr, d) = cost_L(xr + d, d) (:262-287),
//                                                                       stored skewed: the diagonal a right pixel walks is a
//                                                                       column of R, Large_Float where the column is outside
// and every thread scans its two chunk vectors sequentially with the reference's strict '>' (first minimum wins),
// carrying (minimum, argmin) in registers from chunk to chunk: three instructions per cost.  A column outside the image
// is Large_Float: never the minimum (the running minimum starts there).  The two parabola neighbours of each minimum
// are fetched afterwards (four L2 hits per pixel), Large_Float where the reference's cost_local holds it (:277-286).
// Shared memory per CTA is independent of the disparity range (16 KB), so the kernel keeps six CTAs per SM at D = 64
// as at D = 256 -- the first version staged (WT_PX + D - 1) whole columns, 172 KB for a 64-thread CTA at D = 192.
// The right tile's columns are the left tile of the neighbouring CTAs: they come out of L2.
// ---------------------------------------------------------------------------------------------
#define WT_PX 128
#define WT_DC 16
#define WT_LS WT_DC            // row stride of the left tile; quad k of column t is stored at quad k ^ ((t >> 1) & 3): the eight
                               // threads of a 128-bit phase -- eight columns x one quad when scanning, two columns x four quads when
                               // staging -- hit eight different 16-byte bank groups
#define WT_RT ((WT_PX + WT_DC - 1 + WT_PX / 4 - 1) / (WT_PX / 4))   // staging trips of the right tile (32 columns per trip)
#define WT_RS (WT_PX + 3)      // row stride of the right tile: the skewed stores of a warp (columns cj .. cj + 7, four quads) land in 32
                               // different banks: bank = cj + 8 kq + const (with stride 128 it is cj - 4 kq: pairs of lanes collide)

// Side outputs (AUX = true): the cost of the left winner b and the least cost two or more disparities away from it come
// out of the same ascending scan with O(1) state, carried across chunks like (minimum, argmin):
//   pre  min over the indices <= i - 2, fed through the one-step delay q1
//   a strict new minimum at i:   b = i, sec = pre      (everything seen so far that is at least two below i)
//   otherwise, when i >= b + 2:  sec = min(sec, a)     (i = b + 1 is skipped)
// th is b + 2 relative to the chunk, so that the test is one compare against the unrolled chunk index.
struct WtaSecond { float pre, q1, sec; int th; };
__device__ __forceinline__ void wta_second(WtaSecond& s, bool newmin, float a, int k) {
    if (newmin) { s.sec = s.pre; s.th = k + 2; }
    else if (k >= s.th) s.sec = a < s.sec ? a : s.sec;
    s.pre = s.q1 < s.pre ? s.q1 : s.pre;
    s.q1 = a;
}

// AUX = false is the plain kernel; AUX = true keeps one CTA fewer per SM for the four extra registers of the state above
template <bool AUX>
__global__ void __launch_bounds__(WT_PX, AUX ? 5 : 6)
k_wta(AdcDims dm, const float* __restrict__ vol, float* __restrict__ disp_l, float* __restrict__ disp_r, AdcAux aux) {
    __shared__ __align__(16) float tl[WT_PX * WT_LS];
    __shared__ float tr[WT_DC * WT_RS];
    const int pair = blockIdx.z, y = blockIdx.y, x0 = blockIdx.x * WT_PX;
    const int W = dm.W, D = dm.D, Dp = dm.Dp;
    const float* rowv = vol + (size_t)pair * dm.vol_stride + (size_t)y * W * Dp;
    const int t = threadIdx.x;
    const int kq = t & 3, cj = t >> 2;                  // staging role: float4 kq of the chunk, 32 columns per trip
    const float4 LARGE4 = make_float4(ADC_LARGE_F, ADC_LARGE_F, ADC_LARGE_F, ADC_LARGE_F);
    float lbest = ADC_LARGE_F, rbest = ADC_LARGE_F;     // min_cost starts at Large_Float (:209, :266)
    int lbd = -1, rbd = -1;                             // argmin as index d - dmin, -1 = none yet
    WtaSecond s2{ADC_INVALID_F, ADC_INVALID_F, ADC_INVALID_F, 1};
    float4 vl[WT_PX / 32], vr[WT_RT];
    // The loads of chunk c + 1 are issued before chunk c is scanned and land in registers while the scan runs.
    auto fetch = [&](int d0) {
        const bool qin = d0 + 4 * kq < Dp;              // this float4 exists (Dp is a multiple of 4)
        const float* cv = rowv + d0 + 4 * kq;
        const int cb = x0 + dm.dmin + d0;               // image column of column 0 of the right tile
#pragma unroll
        for (int i = 0; i < WT_PX / 32; i++) {          // left tile: columns x0 .. x0 + WT_PX - 1
            const int x = x0 + cj + 32 * i;
            vl[i] = (qin && x < W) ? __ldg(reinterpret_cast<const float4*>(cv + x * Dp)) : LARGE4;
        }
#pragma unroll
        for (int i = 0; i < WT_RT; i++) {               // right tile: column j of the tile is image column cb + j
            const int j = cj + 32 * i, x = cb + j;
            vr[i] = (qin && j < WT_PX + WT_DC - 1 && x >= 0 && x < W) ? __ldg(reinterpret_cast<const float4*>(cv + x * Dp)) : LARGE4;
        }
    };
    fetch(0);
    for (int d0 = 0; d0 < D; d0 += WT_DC) {
        const int dn = min(WT_DC, D - d0);
#pragma unroll
        for (int i = 0; i < WT_PX / 32; i++) {
            *reinterpret_cast<float4*>(tl + (cj + 32 * i) * WT_LS + 4 * (kq ^ ((cj >> 1) & 3))) = vl[i];
        }
#pragma unroll
        for (int i = 0; i < WT_RT; i++) {               // element k of tile column j belongs to right pixel r = j - k
            const int r0 = cj + 32 * i - 4 * kq;
            const float e[4] = {vr[i].x, vr[i].y, vr[i].z, vr[i].w};
#pragma unroll
            for (int c = 0; c < 4; c++) {
                const int r = r0 - c;
                if (r >= 0 && r < WT_PX) tr[(4 * kq + c) * WT_RS + r] = e[c];
            }
        }
        __syncthreads();
        if (d0 + WT_DC < D) fetch(d0 + WT_DC);
        // ---- scans: thread t = left pixel x0 + t and right pixel x0 + t; indices relative to the chunk
        const float* pl = tl + t * WT_LS;
        const int sw = ((t >> 1) & 3) << 2;             // this column's quad swizzle, as a word offset
        const float* pr = tr + t;
        int lk = -1, rk = -1;
        if (dn == WT_DC) {
#pragma unroll
            for (int k4 = 0; k4 < WT_DC; k4 += 4) {
                const float4 a4 = *reinterpret_cast<const float4*>(pl + (k4 ^ sw));
                const float a[4] = {a4.x, a4.y, a4.z, a4.w};
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    const float b = pr[(k4 + j) * WT_RS];
                    const bool nl = lbest > a[j];
                    if (nl) { lbest = a[j]; lk = k4 + j; }
                    if (AUX) wta_second(s2, nl, a[j], k4 + j);
                    if (rbest > b) { rbest = b; rk = k4 + j; }
                }
            }
        } else {
            for (int k = 0; k < dn; k++) {
                const float a = pl[k ^ sw], b = pr[k * WT_RS];
                const bool nl = lbest > a;
                if (nl) { lbest = a; lk = k; }
                if (AUX) wta_second(s2, nl, a, k);
                if (rbest > b) { rbest = b; rk = k; }
            }
        }
        if (lk >= 0) lbd = d0 + lk;
        if (rk >= 0) rbd = d0 + rk;
        if (AUX) s2.th -= WT_DC;
        __syncthreads();
    }
    const int x = x0 + t;
    if (x >= W) return;
    const size_t o = (size_t)pair * dm.N + (size_t)y * W + x;
    {   // left view: a minimum at either end of the range (or none) is Invalid (ADCensusStereo.cpp:224-227)
        float out = ADC_INVALID_F;
        if (lbd > 0 && lbd < D - 1) {
            const float* v = rowv + x * Dp + lbd;
            out = adc_subpixel(__ldg(v - 1), __ldg(v + 1), lbest, dm.dmin + lbd);
        }
        disp_l[o] = out;
        if (AUX) {
            if (aux.cost_best) aux.cost_best[o] = lbest;
            if (aux.cost_second) aux.cost_second[o] = s2.sec;
            if (aux.origin) aux.origin[o] = out == ADC_INVALID_F ? ADC_ORIGIN_WTA_INVALID : 0;
        }
    }
    {   // right view: a minimum at either end gives the integer disparity, not Invalid (:290-293); `best` starts at 0
        // (not dmin) when no column was valid, as in the reference (:271); a parabola neighbour whose column lies
        // outside the image is Large_Float (:277-286)
        float out = 0.0f;
        if (rbd >= 0) {
            const int best = dm.dmin + rbd;
            out = (float)best;
            if (rbd > 0 && rbd < D - 1) {
                const int x1 = x + best - 1, x2 = x + best + 1;
                const float c1 = (x1 >= 0 && x1 < W) ? __ldg(rowv + x1 * Dp + rbd - 1) : ADC_LARGE_F;
                const float c2 = (x2 >= 0 && x2 < W) ? __ldg(rowv + x2 * Dp + rbd + 1) : ADC_LARGE_F;
                out = adc_subpixel(c1, c2, rbest, best);
            }
        }
        disp_r[o] = out;
    }
}

int adc_launch_wta(const AdcParams& P, const AdcWave& w, const float* vol, cudaStream_t st, unsigned long long* launches) {
    dim3 grid((P.dm.W + WT_PX - 1) / WT_PX, P.dm.H, w.S);
    k_wta<false><<<grid, WT_PX, 0, st>>>(P.dm, vol, w.disp_l, w.disp_r, AdcAux{});
    ++*launches;
    return 0;
}

int adc_launch_wta_aux(const AdcParams& P, const AdcWave& w, const float* vol, const AdcAux& aux, cudaStream_t st,
                       unsigned long long* launches) {
    dim3 grid((P.dm.W + WT_PX - 1) / WT_PX, P.dm.H, w.S);
    k_wta<true><<<grid, WT_PX, 0, st>>>(P.dm, vol, w.disp_l, w.disp_r, aux);
    ++*launches;
    return 0;
}
