// k_cost.cu -- stage 1 of the pipeline: gray conversion, 9x7 census transform and the AD-census
// cost volume (reference: cost_computor.cpp:58-121, adcensus_util.cpp:10-53), plus the colour
// difference maps the scanline optimiser consumes (scanline_optimizer.cpp:113-121, 224-235).
#include "adc_common.cuh"

// ---------------------------------------------------------------------------------------------
// gray + census.  One CTA = 32x8 output pixels of one image; the (8+8)x(32+6) gray tile lives in
// shared memory so each gray value is converted once and compared 63 times from on-chip memory.
// Gray is double precision without contraction (r*0.299 + g*0.587 + b*0.114, truncated), which is
// what cost_computor.cpp:69 evaluates; FMA contraction would flip 2933 of the 2^24 inputs.
// ---------------------------------------------------------------------------------------------
#define CT_W 32
#define CT_H 8
#define CT_HX 3
#define CT_HY 4

// (A table of the 3 x 256 possible products, which leaves two double adds per pixel, was measured: the per-CTA copy of the
//  table into shared memory costs more than the three multiplies it saves -- 220 us against 201 us per wave of 32 pairs.)
__device__ __forceinline__ uint8_t gray_of(const uint8_t* __restrict__ px) {
    const double b = (double)__ldg(px), g = (double)__ldg(px + 1), r = (double)__ldg(px + 2);
    const double v = __dadd_rn(__dadd_rn(__dmul_rn(r, 0.299), __dmul_rn(g, 0.587)), __dmul_rn(b, 0.114));
    return (uint8_t)__double2int_rz(v);
}

__global__ void __launch_bounds__(CT_W* CT_H)
k_gray_census(AdcDims dm, const uint8_t* __restrict__ bgr, uint8_t* __restrict__ gray,
              unsigned long long* __restrict__ census, unsigned* __restrict__ bgrx) {
    __shared__ uint8_t tile[CT_H + 2 * CT_HY][CT_W + 2 * CT_HX + 2];
    const int img = blockIdx.z;  // pair*2 + view
    const uint8_t* src = bgr + (size_t)img * dm.N * 3;
    uint8_t* g_out = gray + (size_t)img * dm.N;
    unsigned long long* c_out = census + (size_t)img * dm.N;
    const int x0 = blockIdx.x * CT_W, y0 = blockIdx.y * CT_H;
    const int tid = threadIdx.y * CT_W + threadIdx.x;
    constexpr int TW = CT_W + 2 * CT_HX, TH = CT_H + 2 * CT_HY;
    for (int i = tid; i < TW * TH; i += CT_W * CT_H) {
        const int ty = i / TW, tx = i - ty * TW;
        const int gx = x0 + tx - CT_HX, gy = y0 + ty - CT_HY;
        uint8_t v = 0;
        if (gx >= 0 && gx < dm.W && gy >= 0 && gy < dm.H) v = gray_of(src + ((size_t)gy * dm.W + gx) * 3);
        tile[ty][tx] = v;
    }
    __syncthreads();
    const int x = x0 + threadIdx.x, y = y0 + threadIdx.y;
    if (x >= dm.W || y >= dm.H) return;
    const int tx = threadIdx.x + CT_HX, ty = threadIdx.y + CT_HY;
    const uint8_t centre = tile[ty][tx];
    g_out[(size_t)y * dm.W + x] = centre;
    {   // packed copy of the pixel (B | G<<8 | R<<16) for the kernels that compare colours
        const uint8_t* px = src + ((size_t)y * dm.W + x) * 3;
        bgrx[(size_t)img * dm.N + (size_t)y * dm.W + x] = (unsigned)__ldg(px) | ((unsigned)__ldg(px + 1) << 8) | ((unsigned)__ldg(px + 2) << 16);
    }
    unsigned long long bits = 0ull;
    // border pixels keep 0 and tiny images are skipped entirely (adcensus_util.cpp:12,17-18)
    if (dm.W > 9 && dm.H > 7 && y >= 4 && y < dm.H - 4 && x >= 3 && x < dm.W - 3) {
#pragma unroll
        for (int dy = -CT_HY; dy <= CT_HY; dy++)
#pragma unroll
            for (int dx = -CT_HX; dx <= CT_HX; dx++)
                bits = (bits << 1) | (unsigned long long)(tile[ty + dy][tx + dx] < centre);
    }
    c_out[(size_t)y * dm.W + x] = bits;
}

void adc_launch_gray_census(const AdcParams& P, const AdcWave& w, cudaStream_t st, unsigned long long* launches) {
    dim3 grid((P.dm.W + CT_W - 1) / CT_W, (P.dm.H + CT_H - 1) / CT_H, w.S * 2), block(CT_W, CT_H);
    k_gray_census<<<grid, block, 0, st>>>(P.dm, w.bgr, w.gray, w.census, w.bgrx);
    ++*launches;
}

// ---------------------------------------------------------------------------------------------
// AD-census cost volume.  One thread = one pixel x four consecutive disparities -> one 128-bit
// store; consecutive threads cover consecutive disparity quads of the same pixel, then the next
// pixel, so a warp writes 512 contiguous bytes.  The two exp() factors have tiny integer domains
// (sum of abs differences 0..765, Hamming 0..63): they come from tables built on the host with the
// host's libm expf, evaluated in the reference's order  ((1 - e_ad) + 1) - e_cen
// (cost_computor.cpp:110-117), so the volume is bit-identical to the CPU path by construction.
//
// A thread computes a 4 x 4 block: four neighbouring pixels x0 .. x0 + 3 (x0 a multiple of 4 inside the CTA's segment of
// the row) times four consecutive disparities 4q .. 4q + 3.  Pixel x0 + i at disparity index 4q + j is matched against
// right-image column x0 + i - dmin - 4q - j: the sixteen pairs of the block touch only SEVEN right-image entries (they
// are constant along the diagonals), which sit in two consecutive, 16-byte-aligned vectors of the staged row -- the row
// is staged with an offset that makes that true for every block.  Per block: 2 x 3 128-bit loads of right-image entries
// (packed BGR, low and high census words), 3 of left-image entries (broadcast to the lanes that share the pixels), 32
// table look-ups, four 128-bit stores (a warp writes 2 x 4 runs of 256 contiguous bytes).
// What bounds the kernel is shared-memory bandwidth (one wavefront per clock and SM): version 3 fetched every entry once
// per pair (3 words per cost) and spent 3 wavefronts per AD look-up on bank conflicts -- 7 wavefronts per 32 costs; this
// one needs 4.9.  A CTA computes four consecutive rows of its segment; the tables are staged once per CTA, replicated (x32 for the 64-entry census table: conflict-free;
// x16 for the 766-entry AD table: two lanes per replica) so that the data-dependent look-ups of a warp spread over the
// banks.
// (Measured and rejected in round 2: lanes = 32 consecutive disparities of one pixel -- half the index arithmetic, but
//  32-bit stores and table addresses that differ in every lane: 631 us against 486 us per wave of 32 Cone pairs; one pixel x
//  four disparities per thread with a single 128-bit load per array out of four shifted copies of the row: half the
//  instructions of version 3 and exactly its time, 482 us -- same shared-memory wavefronts.)
// ---------------------------------------------------------------------------------------------
#define CV_AD_REP 16
#define CV_SEG_COLS 928       // columns per CTA at most: longer rows are cut into segments (multiple of 4)

__host__ __device__ inline int cv_pads(int D) { return 4 + ((4 - (D & 3)) & 3); }                  // (D + pads) % 4 == 0, pads >= 4
__host__ __device__ inline int cv_row_len(int Lx, int D) { return (Lx + D + cv_pads(D) + 3) & ~3; }  // staged right-image entries

template <bool EXACT>     // EXACT: D is a multiple of 4, no padding disparities
__global__ void __launch_bounds__(512)
k_cost_volume(AdcDims dm, int gpc, int nseg, int Lx, int rpc, const unsigned* __restrict__ bgrx,
              const unsigned long long* __restrict__ census, float* __restrict__ vol,
              const float* __restrict__ lut_ad, const float* __restrict__ lut_cen) {
    extern __shared__ __align__(16) unsigned char cv_smem[];
    const int pair = blockIdx.y, yb = blockIdx.x / nseg, seg = blockIdx.x - yb * nseg;   // rows yb * rpc .. of segment seg
    const int xa = seg * Lx, xb = min(dm.W, xa + Lx);   // this CTA's columns of row y (xa is a multiple of 4)
    const int Q = dm.Dp >> 2;                           // threads per pixel group
    const int pads = cv_pads(dm.D);
    const int LA = cv_row_len(Lx, dm.D);
    const int span = xb - xa + dm.D - 1;                // right-image columns a pixel of the segment can ask for: entry e is
    const int xr_base = xa - (dm.D - 1) - dm.dmin;      // column xr_base + e (xr = x - dmin - di; x = xa, di = D - 1 is entry 0)
    float* s_ce = reinterpret_cast<float*>(cv_smem);                                      // [64][32]
    float* s_ad = s_ce + 64 * 32;                                                         // [766][CV_AD_REP]
    unsigned* s_rb = reinterpret_cast<unsigned*>(s_ad + 766 * CV_AD_REP);                 // [LA] right image: entry e at position e + pads
    unsigned* s_rl = s_rb + LA;                                                           //      census bits 0..31
    unsigned* s_rh = s_rl + LA;                                                           //      census bits 32..63
    unsigned* s_lb = s_rh + LA;                                                           // [Lx] left image, column xa + i at position i
    unsigned* s_ll = s_lb + Lx;
    unsigned* s_lh = s_ll + Lx;
    const unsigned* left = bgrx + (size_t)pair * 2 * dm.N;
    const unsigned* right = left + (size_t)dm.N;
    const unsigned long long* cen_l = census + (size_t)pair * 2 * dm.N;
    const unsigned long long* cen_r = cen_l + dm.N;
    const int lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < 64 * 8; i += blockDim.x) {              // the tables, once per CTA (128-bit stores)
        const float v = __ldg(lut_cen + (i >> 3));
        reinterpret_cast<float4*>(s_ce)[i] = make_float4(v, v, v, v);
    }
    for (int i = threadIdx.x; i < 766 * (CV_AD_REP / 4); i += blockDim.x) {
        const float v = __ldg(lut_ad + i / (CV_AD_REP / 4));
        reinterpret_cast<float4*>(s_ad)[i] = make_float4(v, v, v, v);
    }
    const int g0 = threadIdx.x / Q, q = threadIdx.x - g0 * Q;
    const float* t_ad = s_ad + (lane & (CV_AD_REP - 1));
    const float* t_ce = s_ce + lane;
    const int ngroups = (xb - xa + 3) >> 2;
    for (int y = yb * rpc; y < min(dm.H, (yb + 1) * rpc); y++) {
        const int row = y * dm.W;
        if (y > yb * rpc) __syncthreads();                // everybody is done with the previous row's entries
        for (int i = threadIdx.x; i < LA; i += blockDim.x) {
            const int e = i - pads, xr = xr_base + e;
            unsigned long long c = 0ull;
            unsigned pix = 0xffffffffu;                 // marker: outside the image
            if (e >= 0 && e < span && xr >= 0 && xr < dm.W) {
                c = __ldg(cen_r + row + xr);
                pix = __ldg(right + row + xr);
            }
            s_rb[i] = pix; s_rl[i] = (unsigned)c; s_rh[i] = (unsigned)(c >> 32);
        }
        for (int i = threadIdx.x; i < Lx; i += blockDim.x) {
            unsigned long long c = 0ull;
            unsigned pix = 0u;
            if (xa + i < xb) { c = __ldg(cen_l + row + xa + i); pix = __ldg(left + row + xa + i); }
            s_lb[i] = pix; s_ll[i] = (unsigned)c; s_lh[i] = (unsigned)(c >> 32);
        }
        __syncthreads();
        float* vrow = vol + (size_t)pair * dm.vol_stride + ((size_t)row + xa) * dm.Dp;
        for (int g = g0; g < (g0 < gpc ? ngroups : 0); g += gpc) {
            // block (i, j): entry e0 + 3 - j + i with e0 = 4g + D - 4 - 4q >= -3; position e0 + pads is a multiple of 4
            const int p0 = 4 * g + dm.D - 4 - 4 * q + pads;
            const uint4 b0 = *reinterpret_cast<const uint4*>(s_rb + p0), b1 = *reinterpret_cast<const uint4*>(s_rb + p0 + 4);
            const uint4 l0 = *reinterpret_cast<const uint4*>(s_rl + p0), l1 = *reinterpret_cast<const uint4*>(s_rl + p0 + 4);
            const uint4 h0 = *reinterpret_cast<const uint4*>(s_rh + p0), h1 = *reinterpret_cast<const uint4*>(s_rh + p0 + 4);
            const uint4 cb = *reinterpret_cast<const uint4*>(s_lb + 4 * g), cl = *reinterpret_cast<const uint4*>(s_ll + 4 * g),
                        ch = *reinterpret_cast<const uint4*>(s_lh + 4 * g);
            const unsigned rb[7] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z};
            const unsigned rl[7] = {l0.x, l0.y, l0.z, l0.w, l1.x, l1.y, l1.z};
            const unsigned rh[7] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z};
            const unsigned lb[4] = {cb.x, cb.y, cb.z, cb.w}, ll[4] = {cl.x, cl.y, cl.z, cl.w}, lh[4] = {ch.x, ch.y, ch.z, ch.w};
    #pragma unroll
            for (int i = 0; i < 4; i++) {
                float out[4];
    #pragma unroll
                for (int j = 0; j < 4; j++) {
                    // branch-free: padding disparities (di >= D) and out-of-image matches compute on whatever the entry holds and
                    // are overwritten by selects -- the per-disparity branches used to cost more than the arithmetic
                    const int c = 3 - j + i;
                    const int sad = min((int)__vsadu4(lb[i], rb[c]), 765);     // |dB| + |dG| + |dR| (4th byte is 0 in both; the marker clamps)
                    const int ham = (__popc(ll[i] ^ rl[c]) + __popc(lh[i] ^ rh[c])) & 63;
                    float v = __fsub_rn(t_ad[sad * CV_AD_REP], t_ce[ham * 32]);
                    v = rb[c] == 0xffffffffu ? 1.0f : v;                        // out-of-image match: cost_computor.cpp:101-104
                    out[j] = (EXACT || 4 * q + j < dm.D) ? v : 0.0f;            // padding disparity, never read as a cost
                }
                if (xa + 4 * g + i < xb)
                    *reinterpret_cast<float4*>(vrow + (size_t)(4 * g + i) * dm.Dp + 4 * q) = make_float4(out[0], out[1], out[2], out[3]);
            }
        }
    }
}

#define CV_SMEM_ATTR (96 * 1024)
static int cv_nseg(int W) { return (W + CV_SEG_COLS - 1) / CV_SEG_COLS; }
static int cv_seg_len(int W) { const int nseg = cv_nseg(W); return (((W + nseg - 1) / nseg) + 3) & ~3; }   // a multiple of 4
static size_t cv_smem_bytes(int Lx, int D) { return (size_t)(64 * 32 + 766 * CV_AD_REP) * 4 + (size_t)3 * cv_row_len(Lx, D) * 4 + (size_t)3 * Lx * 4; }

// at Lx = CV_SEG_COLS and D = 512: 85,680 bytes
size_t adc_cost_smem(const AdcDims& dm, size_t* cap) {
    *cap = CV_SMEM_ATTR;
    return cv_smem_bytes(cv_seg_len(dm.W), dm.D);
}

void adc_launch_cost(const AdcParams& P, const AdcWave& w, float* vol, cudaStream_t st, unsigned long long* launches) {
    const int Q = P.dm.Dp / 4;
    const int nseg = cv_nseg(P.dm.W);
    const int Lx = cv_seg_len(P.dm.W);                                     // columns per segment
    const int groups = Lx / 4;
    int gmax = 512 / Q;                             // pixel groups in flight per CTA
    if (gmax > 32) gmax = 32;
    if (gmax < 1) gmax = 1;
    const int trips = (groups + gmax - 1) / gmax;
    const int gpc = (groups + trips - 1) / trips;   // ... evened out over the trips
    const int threads = (gpc * Q + 31) / 32 * 32;
    const size_t smem = cv_smem_bytes(Lx, P.dm.D);
    static AdcOnce attr_once;
    if (adc_once_needed(attr_once)) {
        cudaFuncSetAttribute(k_cost_volume<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, CV_SMEM_ATTR);
        cudaFuncSetAttribute(k_cost_volume<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, CV_SMEM_ATTR);
        adc_once_done(attr_once);
    }
    const int rpc = 4;                              // rows per CTA: the 57 KB of tables are staged once per four rows
    dim3 grid((P.dm.H + rpc - 1) / rpc * nseg, w.S);
    if (P.dm.D == P.dm.Dp) k_cost_volume<true><<<grid, threads, smem, st>>>(P.dm, gpc, nseg, Lx, rpc, w.bgrx, w.census, vol, w.lut_ad, w.lut_cen);
    else k_cost_volume<false><<<grid, threads, smem, st>>>(P.dm, gpc, nseg, Lx, rpc, w.bgrx, w.census, vol, w.lut_ad, w.lut_cen);
    ++*launches;
}

// ---------------------------------------------------------------------------------------------
// Colour-difference maps for the scanline optimiser: max-channel distance between a pixel and
// its predecessor along x (h) or y (v), for the left and the right image.  A forward pass reads
// map[cur]; a backward pass reads map[pixel it came from] (same two pixels, see k_scanline.cu).
// ---------------------------------------------------------------------------------------------
__global__ void k_diffmaps(AdcDims dm, const uint8_t* __restrict__ bgr, uint8_t* __restrict__ dmap) {
    const int pair = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= dm.N) return;
    const int y = i / dm.W, x = i - y * dm.W;
    uint8_t* out = dmap + (size_t)pair * 4 * dm.N;
#pragma unroll
    for (int v = 0; v < 2; v++) {
        const uint8_t* img = bgr + ((size_t)pair * 2 + v) * dm.N * 3;
        const uchar3 c = adc_load_bgr(img, i);
        out[(size_t)(2 * v) * dm.N + i] = x > 0 ? (uint8_t)adc_colour_dist(c, adc_load_bgr(img, i - 1)) : 0;
        out[(size_t)(2 * v + 1) * dm.N + i] = y > 0 ? (uint8_t)adc_colour_dist(c, adc_load_bgr(img, i - dm.W)) : 0;
    }
}

void adc_launch_diffmaps(const AdcParams& P, const AdcWave& w, cudaStream_t st, unsigned long long* launches) {
    dim3 grid((P.dm.N + 255) / 256, w.S);
    k_diffmaps<<<grid, 256, 0, st>>>(P.dm, w.bgr, w.dmap);
    ++*launches;
}
