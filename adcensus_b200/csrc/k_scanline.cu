// k_scanline.cu -- stage 3: the four chained scanline-optimisation passes
// (reference: scanline_optimizer.cpp:40-61 sequencing, :63-171 horizontal, :173-279 vertical).
//
// One warp owns one scanline (a row for the +-x passes, a column for the +-y passes) and walks it
// serially; the D disparities of a pixel are spread over the 32 lanes, K consecutive ones per
// lane, and live in registers from one step to the next.  Per step the recurrence is
//     L(d) = ( C(d) + min( Lp(d), Lp(d-1)+P1, Lp(d+1)+P1, minLp+P2 ) ) / 2
// (no "- minLp" term, and a "/2": scanline_optimizer.cpp:144-151), with Lp padded by Large_Float
// on both ends and the running minimum taken over the pads too (:96,:107-110).  Neighbour values
// cross lanes through two shuffles; the minimum over d is one REDUX on order-preserving integer
// keys.  Only add/min/exact scalings occur, so the result is bit-identical to the CPU path.
//
// Memory system: everything a step needs that does not depend on the recurrence -- the pixel's
// cost vector (Dp floats) and a small "penalty record" -- is streamed into a per-warp shared
// memory ring with cp.async (LDGSTS), SO_PF steps ahead, so HBM/L2 latency never sits on the
// serial chain and the number of bytes in flight per SM is set by the ring depth, not by
// register scoreboards.
//
// Penalty record.  P1/P2 depend on d1 = Dc(left[p], left[p_prev]) and d2 = Dc(right[xr],
// right[xr_prev]) with xr = x - d - dmin, through (d1 < tso, d2 < tso).  The reference declares d2
// once per pixel (initialised to d1) and only overwrites it while 0 < xr < W-1, so for
// disparities past the valid interval it keeps the value of the last valid one ("sticky d2",
// :116-121).  Closed form: valid d form [lo,hi] = [max(0,x-dmin-(W-2)), min(D-1,x-dmin-1)];
// d<lo -> d1, d in [lo,hi] -> map(x-d-dmin), d>hi -> map(x-hi-dmin), empty interval -> d1.
// k_so_records folds all of that into, per pixel, one word (d1 < tso) and a D-bit string
// (bit d = d2(d) < tso); the bit string is a window of a per-row bit vector of the right image
// stored mirrored, so that increasing d walks increasing bit positions.
#include "adc_common.cuh"

template <int K>
struct Piece { static constexpr int G = (K % 4 == 0) ? 4 : ((K % 2 == 0) ? 2 : 1); static constexpr int NP = K / G; };

template <int K>
__device__ __forceinline__ void ld_vec(const float* p, int lane, int Dp, float (&v)[K]) {   // generic/shared pointer
    constexpr int G = Piece<K>::G, NP = Piece<K>::NP;
#pragma unroll
    for (int j = 0; j < NP; j++) {
        const int d = lane * K + j * G;
        if (d < Dp) {
            if (G == 4) { const float4 t = *reinterpret_cast<const float4*>(p + d); v[j*G] = t.x; v[j*G+1] = t.y; v[j*G+2] = t.z; v[j*G+3] = t.w; }
            else if (G == 2) { const float2 t = *reinterpret_cast<const float2*>(p + d); v[j*G] = t.x; v[j*G+1] = t.y; }
            else v[j] = p[d];
        } else {
#pragma unroll
            for (int g = 0; g < G; g++) v[j * G + g] = 0.f;
        }
    }
}

template <int K>
__device__ __forceinline__ void st_vec(float* __restrict__ p, int lane, int Dp, const float (&v)[K]) {
    constexpr int G = Piece<K>::G, NP = Piece<K>::NP;
#pragma unroll
    for (int j = 0; j < NP; j++) {
        const int d = lane * K + j * G;
        if (d < Dp) {
            if (G == 4) *reinterpret_cast<float4*>(p + d) = make_float4(v[j*G], v[j*G+1], v[j*G+2], v[j*G+3]);
            else if (G == 2) *reinterpret_cast<float2*>(p + d) = make_float2(v[j*G], v[j*G+1]);
            else p[d] = v[j];
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Bit rows of the right image: for variant v in {h-fwd, h-bwd, v-fwd, v-bwd}, bit(xr) of row y says
// whether the colour distance between right(y,xr) and its predecessor along the path is < tso.
// Stored mirrored: bit j of the row holds xr = W-1-j.
// ---------------------------------------------------------------------------------------------
__host__ __device__ inline int so_row_words(int W) { return (W + 31) / 32 + 2; }

__global__ void __launch_bounds__(128)
k_so_bitrows(AdcDims dm, int tso, const uint8_t* __restrict__ dmap, unsigned* __restrict__ bitrows) {
    const int pair = blockIdx.y, y = blockIdx.x;
    const int W = dm.W, rw = so_row_words(W);
    const uint8_t* mh = dmap + ((size_t)pair * 4 + 2) * dm.N;   // right image, distance to (y, x-1)
    const uint8_t* mv = dmap + ((size_t)pair * 4 + 3) * dm.N;   // right image, distance to (y-1, x)
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;  // warp = variant
    unsigned* out = bitrows + (((size_t)pair * 4 + wid) * dm.H + y) * rw;
    for (int w0 = 0; w0 < rw; w0++) {
        const int j = w0 * 32 + lane;
        const int xr = W - 1 - j;
        bool bit = false;
        if (xr > 0 && xr < W - 1) {   // the only positions the reference ever looks at (scanline_optimizer.cpp:120)
            int v;
            if (wid == 0) v = mh[y * W + xr];                 // +x pass: right[xr] vs right[xr-1]
            else if (wid == 1) v = mh[y * W + xr + 1];        // -x pass: right[xr] vs right[xr+1]
            else if (wid == 2) v = y > 0 ? mv[y * W + xr] : 255;            // +y pass: row y vs y-1 (never a path head's successor at y=0)
            else v = y + 1 < dm.H ? mv[(y + 1) * W + xr] : 255;             // -y pass: row y vs y+1
            bit = v < tso;
        }
        const unsigned m = __ballot_sync(0xffffffffu, bit);
        if (lane == 0) out[w0] = m;
    }
}

// per-pixel record for one pass direction: word 0 = (d1 < tso), words 1.. = bit d -> (d2(d) < tso)
__host__ __device__ inline int so_rec_words(int Dp) { return ((1 + (Dp + 31) / 32 + 1) + 3) / 4 * 4; }

// (one launch writes the records of all four pass directions, blockIdx.z = direction)
__global__ void __launch_bounds__(256)
k_so_records(AdcDims dm, int tso, const uint8_t* __restrict__ dmap,
             const unsigned* __restrict__ bitrows, unsigned* __restrict__ rec) {
    const int pair = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= dm.N) return;
    const int sx = blockIdx.z == 0 ? 1 : (blockIdx.z == 1 ? -1 : 0);
    const int sy = blockIdx.z == 2 ? 1 : (blockIdx.z == 3 ? -1 : 0);
    const int W = dm.W, D = dm.D, dmin = dm.dmin;
    const int y = i / W, x = i - y * W;
    const bool fwd = (sx + sy) > 0;
    const int pstep = sx + sy * W;
    const int variant = sx ? (fwd ? 0 : 1) : (fwd ? 2 : 3);
    const int rw = so_row_words(W), nrec = so_rec_words(dm.Dp);
    unsigned* out = rec + (((size_t)pair * 4 + variant) * dm.N + i) * nrec;
    // d1: this pixel vs the one the path came from (undefined for path heads, which never use it)
    const uint8_t* ml = dmap + ((size_t)pair * 4 + (sx ? 0 : 1)) * dm.N;
    const int pi_from = i - pstep;
    int d1 = 0;
    if (fwd) d1 = ml[i];
    else if (pi_from >= 0 && pi_from < dm.N) d1 = ml[pi_from];
    const unsigned a1 = d1 < tso ? 0xffffffffu : 0u;
    const int lo = max(0, x - dmin - (W - 2));
    const int hi = min(D - 1, x - dmin - 1);
    const unsigned* row = bitrows + (((size_t)pair * 4 + variant) * dm.H + y) * rw;
    const int j0 = W - 1 - x + dmin;           // bit position of d = 0  (xr = x - dmin)
    auto window = [&](int d0) -> unsigned {     // bits d0..d0+31 of the string, 0 where out of the row
        const int j = j0 + d0;                   // |j| < W + D + 64: plain int
        const int wlo = j >> 5;                  // arithmetic shift = floor division also for negative j
        const int sh = j & 31;
        const unsigned a = (wlo >= 0 && wlo < rw) ? row[wlo] : 0u;
        const unsigned b = (wlo + 1 >= 0 && wlo + 1 < rw) ? row[wlo + 1] : 0u;
        return __funnelshift_r(a, b, sh);
    };
    unsigned fill_hi = a1;
    if (lo <= hi) fill_hi = (window(hi) & 1u) ? 0xffffffffu : 0u;
    const int nw = (dm.Dp + 31) / 32 + 1;
    auto word = [&](int w0) -> unsigned {
        if (lo > hi) return a1;
        const int d0 = w0 * 32;
        const unsigned raw = window(d0);
        // masks of the bits with d < lo and d > hi inside this word
        const unsigned m_lo = lo <= d0 ? 0u : (lo >= d0 + 32 ? 0xffffffffu : ((1u << (lo - d0)) - 1u));
        const unsigned m_hi = hi >= d0 + 31 ? 0u : (hi < d0 ? 0xffffffffu : ~((2u << (hi - d0)) - 1u));
        return (raw & ~m_lo & ~m_hi) | (a1 & m_lo) | (fill_hi & m_hi);
    };
    if (nrec == 4) {   // D <= 64: the whole record is one 128-bit store
        *reinterpret_cast<uint4*>(out) = make_uint4(a1, word(0), nw > 1 ? word(1) : 0u, nw > 2 ? word(2) : 0u);
        return;
    }
    out[0] = a1;
    for (int w0 = 0; w0 < nw; w0++) out[1 + w0] = word(w0);
    for (int w0 = 1 + nw; w0 < nrec; w0++) out[w0] = 0u;
}

// ---------------------------------------------------------------------------------------------
// The serial kernel.  A group of LPS lanes (8, 16 or 32) owns one scanline and keeps K = Dp/LPS
// consecutive disparities per lane, so a warp advances 32/LPS neighbouring scanlines in lockstep.
// Fewer lanes per line = more disparities per lane = the per-step bookkeeping (barriers, copy
// issue, neighbour shuffles, the min butterfly) is amortised over more cost values; the kernel
// was issue-bound with 2 values per lane.  For the +-y passes the lines of a warp are adjacent
// columns, i.e. one contiguous 32/LPS * Dp * 4-byte run per step.
#define SO_WARPS 4
#define SO_PF 8      // steps of input kept in flight per line

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

// Bulk asynchronous copies (the TMA engine's 1-D form, cp.async.bulk) completing on an mbarrier: ONE instruction moves a
// pixel's whole cost vector into the ring slot, where the cp.async form needs Dp/4 16-byte copies spread over the lanes.
__device__ __forceinline__ unsigned so_smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(unsigned dst, const void* src, unsigned bytes, unsigned bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
    unsigned ok, spins = 0;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
        if (!ok && ++spins > (1u << 24)) __trap();   // a copy that never completes is a bug: fail the launch instead of hanging the device
    } while (!ok);
}

template <int K, int LPS, bool FULL, bool BULK>   // FULL: D == LPS*K, every lane's K values are real disparities (no padding logic)
                                                  // BULK: ring slots filled by cp.async.bulk + mbarrier (one lane per line issues), else by cp.async
__global__ void __launch_bounds__(SO_WARPS * 32)
k_scanline(AdcParams P, const float* __restrict__ src, float* __restrict__ dst,
           const unsigned* __restrict__ rec, int sx, int sy) {
    constexpr int PF = SO_PF;
    constexpr int LPW = 32 / LPS;               // lines per warp
    // SWZ: a lane's eight costs are two 16-byte chunks 32 bytes apart, so the eight lanes of a 128-bit load phase would hit
    // four bank groups twice; the cp.async fill therefore stores chunk c at position c ^ ((c >> 3) & 1) and the two loads of
    // lane gl read positions 2gl + b and 2gl + 1 - b, b = (gl >> 2) & 1: eight different bank groups per phase.
    constexpr bool SWZ = FULL && K == 8 && !BULK;
    extern __shared__ __align__(16) unsigned char so_smem[];
    const AdcDims& dm = P.dm;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int sub = lane / LPS, gl = lane % LPS;   // line within the warp, lane within the line's group
    const int line = (blockIdx.x * SO_WARPS + wid) * LPW + sub;
    const int pair = blockIdx.y;
    const int n_lines = sx ? dm.H : dm.W, n_steps = sx ? dm.W : dm.H;
    const bool live = line < n_lines;            // dead groups run along (uniform control flow) but move no data
    // FULL: D == Dp == K * LPS is known at compile time, and with it every chunk count, slot size and stride below
    const int W = dm.W, D = FULL ? K * LPS : dm.D, Dp = FULL ? K * LPS : dm.Dp;
    const int pstep = sx + sy * W;               // signed pixel stride along the path
    const int nrec = so_rec_words(Dp);
    const int cost_chunks = Dp >> 2, rec_chunks = nrec >> 2;      // 16-byte chunks per step
    const int slot_bytes = (Dp + nrec) * 4;
    // Ring: PF slots per WARP; a slot holds the cost vectors of the warp's LPW lines back to back, then their records, so
    // that for the +-y passes (the lines are adjacent columns = adjacent memory) ONE bulk copy fills all of them.
    unsigned char* wring = so_smem + (size_t)(wid * PF) * LPW * slot_bytes;
    const int cost_off = sub * Dp * 4, rec_off = LPW * Dp * 4 + sub * nrec * 4;    // this line's part of a slot
    const float* S = src + (size_t)pair * dm.vol_stride;
    float* O = dst + (size_t)pair * dm.vol_stride;
    const int variant = sx ? (sx > 0 ? 0 : 1) : (sy > 0 ? 2 : 3);
    const unsigned* R = rec + ((size_t)pair * 4 + variant) * dm.N * nrec;

    const int x0 = sx ? (sx > 0 ? 0 : W - 1) : line;
    const int y0 = sy ? (sy > 0 ? 0 : dm.H - 1) : line;
    long long pi = (long long)y0 * W + x0;
    if (!live) pi = 0;
    const int line0 = (blockIdx.x * SO_WARPS + wid) * LPW;                        // first line of this warp
    const int nlive = min(LPW, max(0, n_lines - line0));                          // its lines that exist
    // BULK: one mbarrier per (warp, slot), behind the rings of all warps
    const unsigned bar0 = so_smem_u32(so_smem + (size_t)SO_WARPS * PF * LPW * slot_bytes) + (unsigned)(wid * PF) * 8u;
    if (BULK) {
        if (lane == 0) {
#pragma unroll
            for (int j = 0; j < PF; j++) mbar_init(bar0 + 8u * j, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
    }

    // BULK producers: for the +-y passes lane 0 fills the whole slot with two copies (the warp's lines are adjacent columns);
    // for the +-x passes lane l fills line l's part (its lines are different image rows).  Each keeps the addresses of the
    // NEXT step to fetch and advances them by a constant -- prefetch() is called for consecutive steps 1, 2, 3, ...
    const bool producer = BULK && nlive > 0 && (sy ? lane == 0 : lane < nlive);
    const int pline = sy ? 0 : lane;                                              // producer lane -> line of the warp
    const long long pp1 = sy ? ((long long)y0 + sy) * W + line0 : (long long)(line0 + pline) * W + x0 + sx;   // its pixel at step 1
    const float* pcs = S + (producer ? (size_t)pp1 * Dp : 0);
    const unsigned* prs = R + (producer ? (size_t)pp1 * nrec : 0);
    const long long dcs = (long long)pstep * Dp, drs = (long long)pstep * nrec;
    const unsigned pb_c = (unsigned)((sy ? nlive : 1) * Dp * 4), pb_r = (unsigned)((sy ? nlive : 1) * nrec * 4);
    const unsigned po_c = (unsigned)(pline * Dp * 4), po_r = (unsigned)(LPW * Dp * 4 + pline * nrec * 4);

    auto prefetch = [&](int step) {   // issue the copies of `step` into its ring slot (no commit)
        unsigned char* slot = wring + (size_t)(step % PF) * LPW * slot_bytes;
        if (BULK) {   // (the slot's previous contents were read, and fenced against the async proxy, by every lane before the __syncwarp preceding this call)
            const unsigned bar = bar0 + 8u * (unsigned)(step % PF), dst0 = so_smem_u32(slot);
            if (lane == 0 && nlive > 0) mbar_expect_tx(bar, (unsigned)(nlive * slot_bytes));
            if (!sy) __syncwarp();          // the transaction count is armed before another lane's copy can complete on it
            if (producer) {
                bulk_g2s(dst0 + po_c, pcs, pb_c, bar);
                bulk_g2s(dst0 + po_r, prs, pb_r, bar);
                pcs += dcs; prs += drs;
            }
            return;
        }
        if (!live) return;
        const long long p = (long long)y0 * W + x0 + (long long)step * pstep;
        const float* cs = S + (size_t)p * Dp;
        const unsigned* rs = R + (size_t)p * nrec;
        for (int c = gl; c < cost_chunks; c += LPS) cp_async16(slot + cost_off + (SWZ ? (c ^ ((c >> 3) & 1)) : c) * 16, cs + c * 4);
        for (int c = gl; c < rec_chunks; c += LPS) cp_async16(slot + rec_off + c * 16, rs + c * 4);
    };

    bool valid[K];
#pragma unroll
    for (int k = 0; k < K; k++) valid[k] = FULL || (gl * K + k) < D;

    // start the pipeline, then handle the path head: L = C  (scanline_optimizer.cpp:99-100)
#pragma unroll
    for (int j = 1; j <= PF; j++) {
        if (j < n_steps) prefetch(j);
        if (!BULK) cp_async_commit();   // one group per step, empty groups keep the count uniform
    }
    float L[K];
    {
        const float* head = S + (size_t)pi * Dp;
#pragma unroll
        for (int k = 0; k < K; k++) {
            const int d = gl * K + k;
            L[k] = (live && d < Dp) ? __ldg(head + d) : 0.f;
        }
    }
    if (live) st_vec<K>(O + (size_t)pi * Dp, gl, Dp, L);
    float minL = ADC_LARGE_F;
#pragma unroll
    for (int k = 0; k < K; k++) {
        if (!valid[k]) L[k] = ADC_LARGE_F;
        minL = fminf(minL, L[k]);
    }
#pragma unroll
    for (int o = LPS / 2; o >= 1; o >>= 1) minL = fminf(minL, __shfl_xor_sync(0xffffffffu, minL, o));

    const int bit0 = gl * K;   // first disparity of this lane inside the record's bit string
    for (int step = 1; step < n_steps; step++) {
        if (BULK) {                  // the k-th use of a slot completes phase k of its mbarrier: steps step, step + PF, ...
            if (nlive > 0) mbar_wait(bar0 + 8u * (unsigned)(step % PF), (unsigned)((step / PF - (step % PF == 0 ? 1 : 0)) & 1));
        } else {
            cp_async_wait<PF - 1>(); // the group of `step` has landed (for this lane's copies)
            __syncwarp();            // ... and for every other lane's
        }
        const unsigned char* slot = wring + (size_t)(step % PF) * LPW * slot_bytes;
        float C[K];
        if (SWZ) {
            const int b = (gl >> 2) & 1;
            const float4 c0 = *reinterpret_cast<const float4*>(slot + cost_off + (2 * gl + b) * 16);
            const float4 c1 = *reinterpret_cast<const float4*>(slot + cost_off + (2 * gl + 1 - b) * 16);
            C[0] = c0.x; C[1] = c0.y; C[2] = c0.z; C[3] = c0.w;
            C[4 % K] = c1.x; C[5 % K] = c1.y; C[6 % K] = c1.z; C[7 % K] = c1.w;
        } else ld_vec<K>(reinterpret_cast<const float*>(slot + cost_off), gl, Dp, C);
        const unsigned* rw = reinterpret_cast<const unsigned*>(slot + rec_off);
        const bool a1 = rw[0] != 0u;
        const unsigned bits = __funnelshift_r(rw[1 + (bit0 >> 5)], rw[2 + (bit0 >> 5)], bit0 & 31);
        // Everyone has read the slot before it is refilled.  The refill of a BULK ring is a write of the ASYNC proxy (the
        // TMA engine), the reads above went through the generic proxy: each lane orders its reads against that proxy
        // before the barrier -- without the proxy fence about one pair in four of a loaded GPU came out wrong.
        if (BULK) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (step + PF < n_steps) prefetch(step + PF);
        if (!BULK) cp_async_commit();
        pi += pstep;

        const float up = __shfl_up_sync(0xffffffffu, L[K - 1], 1, LPS);
        const float down = __shfl_down_sync(0xffffffffu, L[0], 1, LPS);
        const float left_in = gl == 0 ? ADC_LARGE_F : up;
        const float right_in = gl == LPS - 1 ? ADC_LARGE_F : down;
        // the three penalty classes of this pixel's left-image term (scanline_optimizer.cpp:129-141)
        const float P1a = a1 ? P.p1 : P.p1_4, P1b = a1 ? P.p1_4 : P.p1_10;   // d2 < tso  /  d2 >= tso
        const float P2a = a1 ? P.p2 : P.p2_4, P2b = a1 ? P.p2_4 : P.p2_10;
        const float m4a = __fadd_rn(minL, P2a), m4b = __fadd_rn(minL, P2b);

        float Ln[K];
        float mn = ADC_LARGE_F;
#pragma unroll
        for (int k = 0; k < K; k++) {
            const bool a2 = (bits >> k) & 1u;
            const float P1 = a2 ? P1a : P1b;
            const float l1 = L[k];
            const float l2 = __fadd_rn(k > 0 ? L[k - 1] : left_in, P1);
            const float l3 = __fadd_rn(k < K - 1 ? L[k + 1] : right_in, P1);
            const float l4 = a2 ? m4a : m4b;
            float v = __fadd_rn(C[k], fminf(fminf(l1, l2), fminf(l3, l4)));
            v = __fmul_rn(v, 0.5f);
            Ln[k] = v;
            if (valid[k]) mn = fminf(mn, v);
        }
        if (live) st_vec<K>(O + (size_t)pi * Dp, gl, Dp, Ln);
#pragma unroll
        for (int k = 0; k < K; k++) L[k] = valid[k] ? Ln[k] : ADC_LARGE_F;
#pragma unroll
        for (int o = LPS / 2; o >= 1; o >>= 1) mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        minL = mn;
    }
    if (!BULK) cp_async_wait<0>();
}

#define SO_SMEM_ATTR (160 * 1024)
// ring (+ mbarriers) of one CTA; at Dp = 512 (one line per warp, bulk ring): 68,352 bytes
static size_t so_smem_bytes(int Dp, int LPS, bool bulk) {
    const int slot_bytes = (Dp + so_rec_words(Dp)) * 4;
    return (size_t)SO_WARPS * SO_PF * ((size_t)(32 / LPS) * slot_bytes + (bulk ? 8 : 0));
}
// lanes per line: as few as keep K = ceil(Dp / lanes) <= 8, a whole warp beyond Dp = 256 (K = 9 .. 16)
static int so_lanes_per_line(int Dp) { return Dp <= 64 ? 8 : (Dp <= 128 ? 16 : 32); }

size_t adc_scanline_smem(const AdcDims& dm, size_t* cap) {
    *cap = SO_SMEM_ATTR;
    const int LPS = so_lanes_per_line(dm.Dp);
    return so_smem_bytes(dm.Dp, LPS, LPS == 32);
}

template <int K, int LPS, bool FULL, bool BULK>
static int launch_scanline_kf(const AdcParams& P, const AdcWave& w, const float* src, float* dst, int sx, int sy,
                             cudaStream_t st) {
    constexpr int LPW = 32 / LPS;
    const int n_lines = sx ? P.dm.H : P.dm.W;
    const size_t smem = so_smem_bytes(P.dm.Dp, LPS, BULK);
    static AdcOnce attr_once;
    if (adc_once_needed(attr_once)) {
        cudaFuncSetAttribute(k_scanline<K, LPS, FULL, BULK>, cudaFuncAttributeMaxDynamicSharedMemorySize, SO_SMEM_ATTR);
        adc_once_done(attr_once);
    }
    const int lines_per_block = SO_WARPS * LPW;
    dim3 grid((n_lines + lines_per_block - 1) / lines_per_block, w.S);
    k_scanline<K, LPS, FULL, BULK><<<grid, SO_WARPS * 32, smem, st>>>(P, src, dst, w.so_rec, sx, sy);
    return 0;
}

// Which way a pass fills its ring.  Measured on B200 per pass of a wave (x / y direction), cp.async vs bulk:
//   8 lanes per line  (Cone, D = 64):        582 / 521 us  vs  592 / 537 us
//   16 lanes per line (1242x375, D = 128):   2.67 / 2.44 ms vs 2.68 / 2.46 ms
//   32 lanes per line (1920x1080, D = 192):  6.61 / 6.86 ms vs 6.44 / 6.32 ms
// A bulk copy costs ~20 issue slots (uniform-register set-up, lane election) and every refill needs a proxy fence; it pays
// when one copy moves a whole warp's step (a single line of D > 128 disparities), not when a warp steps four short lines.
template <int K, int LPS>
static int launch_scanline_k(const AdcParams& P, const AdcWave& w, const float* src, float* dst, int sx, int sy,
                             cudaStream_t st) {
    constexpr bool bulk = LPS == 32;
    if (P.dm.D == K * LPS) return launch_scanline_kf<K, LPS, true, bulk>(P, w, src, dst, sx, sy, st);
    return launch_scanline_kf<K, LPS, false, bulk>(P, w, src, dst, sx, sy, st);
}

void adc_launch_so_bitrows(const AdcParams& P, const AdcWave& w, cudaStream_t st, unsigned long long* launches) {
    dim3 grid(P.dm.H, w.S);
    k_so_bitrows<<<grid, 128, 0, st>>>(P.dm, P.tso, w.dmap, w.so_bitrows);
    dim3 rgrid((P.dm.N + 255) / 256, w.S, 4);
    k_so_records<<<rgrid, 256, 0, st>>>(P.dm, P.tso, w.dmap, w.so_bitrows, w.so_rec);
    *launches += 2;
}

int adc_launch_scanline(const AdcParams& P, const AdcWave& w, const float* src, float* dst, int sx, int sy,
                        cudaStream_t st, unsigned long long* launches) {
    // lanes per line: see so_lanes_per_line (Dp is a multiple of 4)
    const int Dp = P.dm.Dp;
    int rc = 1;
#define SO_GO(KK, LL) rc = launch_scanline_k<KK, LL>(P, w, src, dst, sx, sy, st)
    if (Dp <= 64) {            // 8 lanes per line
        switch ((Dp + 7) / 8) { case 1: SO_GO(1, 8); break; case 2: SO_GO(2, 8); break; case 3: SO_GO(3, 8); break; case 4: SO_GO(4, 8); break;
                                case 5: SO_GO(5, 8); break; case 6: SO_GO(6, 8); break; case 7: SO_GO(7, 8); break; default: SO_GO(8, 8); }
    } else if (Dp <= 128) {    // 16 lanes per line
        switch ((Dp + 15) / 16) { case 5: SO_GO(5, 16); break; case 6: SO_GO(6, 16); break; case 7: SO_GO(7, 16); break; default: SO_GO(8, 16); }
    } else if (Dp <= 256) {    // a whole warp per line
        switch ((Dp + 31) / 32) { case 5: SO_GO(5, 32); break; case 6: SO_GO(6, 32); break; case 7: SO_GO(7, 32); break; default: SO_GO(8, 32); }
    } else if (Dp <= 512) {    // a whole warp per line, 9 .. 16 disparities per lane (engines created with a wide range limit)
        switch ((Dp + 31) / 32) { case 9: SO_GO(9, 32); break; case 10: SO_GO(10, 32); break; case 11: SO_GO(11, 32); break;
                                  case 12: SO_GO(12, 32); break; case 13: SO_GO(13, 32); break; case 14: SO_GO(14, 32); break;
                                  case 15: SO_GO(15, 32); break; default: SO_GO(16, 32); }
    } else return 1;           // D > 512 not supported
#undef SO_GO
    ++*launches;
    return rc;
}

size_t adc_so_rec_bytes(const AdcDims& dm) { return (size_t)4 * dm.N * so_rec_words(dm.Dp) * 4; }   // four pass directions
size_t adc_so_bitrow_bytes(const AdcDims& dm) { return (size_t)4 * dm.H * so_row_words(dm.W) * 4; }
