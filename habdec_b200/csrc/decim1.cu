// K1 -- stage-1 FIR decimator, the HBM-bound kernel of the path.
//
// Replaces habdec::Decimator<complex<float>,float>::operator() for the first
// decimation stage (reference: code/Decoder/Decimator.h:99-146, driven from
// code/Decoder/Decoder.h:440-447 with the tap tables chosen at :286-320):
//
//     y[k] = sum_{t=0}^{T-1} x[k*M - (T-1) + t] * h[t]        (x = [history | input])
//
// B200 design (not a translation of the CPU loop):
//  * a WARP is the unit of work.  It owns a "stretch" of consecutive output samples of one
//    channel and streams the matching input window exactly once, HBM -> shared memory, with
//    1-D TMA bulk copies (cp.async.bulk + mbarrier complete_tx) into a private ring of
//    pieces; no thread ever issues a global load for samples, so memory-level parallelism
//    is set by the ring depth, not by occupancy or registers.
//  * polyphase mapping: the input is cut into 64-sample superblocks that END on an output
//    sample; lane l always sees phase l and l+32 of every superblock (two conflict-free
//    LDS.64), so its 2*NLIVE taps live in registers for the whole kernel.  Every lane keeps
//    NLIVE sliding complex accumulators (one per output whose window overlaps the current
//    superblock); each loaded sample is used for T/M (5.4 .. 6.8) FMAs straight from
//    registers.  Completed outputs are lane-partials: 16 of them are transposed through a
//    padded shared tile and summed (LDS.128 + packed FADD2), so the cross-lane reduction costs
//    ~1 LDS + 1.5 FADD2 per superblock instead of a shuffle tree per output.
//  * no tensor cores: complex-by-real FIR taps on a per-channel stream are not a dense
//    contraction (north star), the kernel is bound by the 8 B/sample HBM read.
//
// Summation order differs from the reference's sequential t-loop (lane-partials + tree),
// so results match to ~1e-7 relative, inside the 1e-5 relative-L2 budget of the north star.
#include "hbd_common.cuh"
#include "decim1.cuh"
#include "iq_format.cuh"
#include <algorithm>

namespace hbd {

// ---- small PTX wrappers -------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async()
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    uint32_t done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!done);
}
// global -> shared bulk copy (TMA, 1-D), completion counted in bytes on `bar`
__device__ __forceinline__ void tma_load_1d(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// The same copy with an L2 eviction-priority hint.  K1 streams 2 GB per call through a 126 MB L2 exactly once; marked
// evict-first, those lines go before the ~150 MB the tail kernel re-reads a moment later (stage-1 outputs, low-pass
// queue, slicer queue, channel state), which then mostly hit L2 instead of competing with K1 for HBM.
__device__ __forceinline__ uint64_t l2_policy_evict_first()
{
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void tma_load_1d_hint(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar, uint64_t policy)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
                 : "memory");
}
#ifndef HBD_K1_EVICT_FIRST
#define HBD_K1_EVICT_FIRST 1
#endif

// ---- compile-time geometry of one (M, T) decimator ---------------------------------------------------------
#ifndef HBD_K1_STAGES
#define HBD_K1_STAGES 2
#endif
#ifndef HBD_K1_PSB_MIN
#define HBD_K1_PSB_MIN 12
#endif
template <int M, int T, int PSBMIN = HBD_K1_PSB_MIN>
struct Geo {
    static constexpr int SB    = 64;                   // samples per superblock
    static constexpr int NOUT  = SB / M;               // outputs ending inside one superblock
    static constexpr int NLIVE = (T + SB - 1) / M;     // outputs whose window overlaps a superblock
    static constexpr int RAMP  = 1 + (T - 1 - M) / SB; // superblocks needed before the first owned one
    static constexpr int gcd_(int a, int b) { return b ? gcd_(b, a % b) : a; }
    static constexpr int U     = NLIVE / gcd_(NLIVE, NOUT);       // accumulator rotation period (superblocks)
    static constexpr int RAMP_GROUPS = (RAMP + U - 1) / U;        // ramp-in walked as whole groups of U
    static constexpr int PSB   = U * ((PSBMIN + U - 1) / U); // superblocks per ring piece (multiple of U)
    static constexpr int GROUPS_PER_PIECE = PSB / U;
    static constexpr int PIECE_SAMPLES = PSB * SB;
    static constexpr int PIECE_BYTES   = (PIECE_SAMPLES + 2) * 8; // +2: 16-byte alignment slack on both sides
    // cross-lane reduction tile: one row per completed output, 32 lane-partials (+1 pad) per row
    static constexpr int RED_ROWS = (NOUT == 1) ? PSB : 16;
    static_assert(SB % M == 0, "M must divide 64");
    static_assert(T - 1 >= M, "taps shorter than the decimation factor are not handled by this kernel");
    static_assert(RED_ROWS <= 16, "reduction tile maps (row, re/im) onto the 32 lanes");
};

constexpr int kStages   = HBD_K1_STAGES; // ring depth per warp
constexpr int kRedPitch = 36;            // float2 per row: 16-byte aligned rows, 32 B mod 128 B (see reduce_rows)

#ifndef HBD_K1_RED_IN_RING
#define HBD_K1_RED_IN_RING 1
#endif
// NOUT == 1 (the /64 first stage): the reduction tile of a piece lives INSIDE the ring slot being consumed -- row b
// (288 B) is written after superblock b (512 B) of the slot has been read, so it only ever covers consumed samples, and
// the tile is summed before the slot is handed back to the TMA.  That takes 27 KB per CTA off K1's footprint, which is
// what lets a third tail CTA (or a second FFT CTA) co-reside with K1 on an SM.
//
// Integer input (GRAN = 16 B / sample size > 2): a slot still holds a whole piece as cf32 (boundary pieces are widened in
// place), and the TMA puts the integers RIGHT-aligned into it, at kIntOff.  Widening forward in batches of 32 samples is then
// safe in place (cf32 of samples < s ends at 8 s <= kIntOff + s * bytes, where the integers of sample s start), and the
// reduction rows (288 B per consumed 64 samples) stay below the integers not yet read.
template <int M, int T, int PSBMIN = HBD_K1_PSB_MIN, int STAGES = kStages, int GRAN = 2>
struct WarpSmem {
    using G = Geo<M, T, PSBMIN>;
    static constexpr bool kRedInRing = HBD_K1_RED_IN_RING && G::NOUT == 1 && G::PSB * kRedPitch * 8 <= G::PSB * 64 * 8;
    static constexpr int kSlotSamples = G::PIECE_SAMPLES + GRAN;               // + alignment slack on both sides
    static constexpr int kIntOff = (8 - 16 / GRAN) * kSlotSamples;             // byte offset of the integers (GRAN > 2)
    static_assert(GRAN != 2 || kSlotSamples * 8 == G::PIECE_BYTES, "cf32 slot layout");
    alignas(16) unsigned char ring[STAGES][kSlotSamples * 8];
    alignas(16) float2 red[kRedInRing ? 1 : G::RED_ROWS][kRedPitch];
    alignas(8) uint64_t full[STAGES];
};
// The NCO variant is bound by instruction issue, not by bytes in flight (a wideband capture row is re-read from L2 by every
// channel): more warps (14 instead of 8) with a two-deep ring hide the latency of its longer dependent chains.  Measured on
// 4096 channels of one 20 MS/s capture (tools/bench_wideband.py): 8 warps x 3 stages (round 1) 0.560 ms, 16 warps x 3 stages of
// half-size pieces 0.448 ms (the per-piece overhead doubles), 12 x 2 0.424 ms, 14 x 2 0.384 ms.
#ifndef HBD_NCO_WARPS
#define HBD_NCO_WARPS 14
#endif
#ifndef HBD_NCO_PSB
#define HBD_NCO_PSB 12
#endif
#ifndef HBD_NCO_STAGES
#define HBD_NCO_STAGES 2
#endif
template <bool NCO> struct K1Cfg {
    static constexpr int kWarps = NCO ? HBD_NCO_WARPS : kDecimWarps;
    static constexpr int kPsbMin = NCO ? HBD_NCO_PSB : HBD_K1_PSB_MIN;
    static constexpr int kSt = NCO ? HBD_NCO_STAGES : kStages;
};

// taps for lane position P (0..63) and live output j (1..NLIVE): t = T - M*j + P
template <int M, int T>
__device__ __forceinline__ float tap_for(const float* __restrict__ taps, int j, int P)
{
    const int t = T - M * j + P;
    return (t >= 0 && t < T) ? __ldg(taps + t) : 0.0f;
}

// Sum the 32 lane-partials of up to 16 staged outputs and store the ones whose output index lies in [k_lo, k_hi).
// Row r of the tile is output k_first + r.  Lane = 2*row + h: it adds the 16 partials held in the row's float4 slots
// 2i + h (8 LDS.128, packed FADD2 tree), the two halves meet through one shuffle.  The row pitch of 36 float2
// (288 B = 32 B mod 128 B) makes the eight lanes of every LDS.128 phase hit eight different 16-byte bank groups.
__device__ __forceinline__ void reduce_rows(const float2 (*red)[kRedPitch], int rows, int k_first, int k_lo, int k_hi,
                                            float2* __restrict__ out, int lane)
{
    __syncwarp();
    const int row = lane >> 1, h = lane & 1;
    const float4* src = reinterpret_cast<const float4*>(&red[min(row, rows - 1)][0]) + h;  // lanes beyond `rows` re-read the last row
    float2 s[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const float4 v = src[2 * i];
        s[i] = cadd2(make_float2(v.x, v.y), make_float2(v.z, v.w));
    }
    const float2 a = cadd2(cadd2(s[0], s[1]), cadd2(s[2], s[3])), b = cadd2(cadd2(s[4], s[5]), cadd2(s[6], s[7]));
    float2 t = cadd2(a, b);
    t.x += __shfl_xor_sync(0xffffffffu, t.x, 1);
    t.y += __shfl_xor_sync(0xffffffffu, t.y, 1);
    const int k = k_first + row;
    if (h == 0 && row < rows && k >= k_lo && k < k_hi) out[k] = t;
    __syncwarp();
}

// ---- fused NCO (K0 inside K1) ---------------------------------------------------------------------------------------
// phasor(j) = cf32( E[j >> 12] * S1[(j >> 6) & 63] ) (x) cf32( S2[j & 63] ),  E[B] = cis(ph0 + 4096 B inc), S1[a] = cis(64 a inc),
// S2[b] = cis(b inc), cis(p) = exp(-2 pi i frac(p)): every factor is an exact float64 sincospi, E * S1 is a float64
// product (once per 64 samples), the last product is float with a fixed operation order, so the value depends on j only
// (ramp-in overlap of two spans, the carry written for the next call and the samples filtered in this call all see the
// same number).  It differs from the directly evaluated, once-rounded phasor of the oracle (pyoracle.premix) by at most
// ~1.5e-7 relative -- the size of the FIR's own float rounding, two orders below the 1e-5 stage tolerance.  (A float64
// product per sample costs 4 FP64 operations + 2 conversions and made this kernel 2.3x slower than the plain K1.)
struct NcoWarpSmem {
    double2 s1[64];       // S1[a] = cis(64 a inc)
    float2 s2[64];        // cf32(S2[b]), S2[b] = cis(b inc)
    double2 e[32];        // E[ebase .. ebase+31]
    float4 pq[16];        // cf32(E * S1) of the 64-sample groups a ring piece touches, as (re, re, im, im): both packed operands of a product
};
__device__ __forceinline__ double2 nco_cis(double ph)
{
    ph -= floor(ph);
    double sn, cs;
    sincospi(-2.0 * ph, &sn, &cs);
    return make_double2(cs, sn);
}
__device__ __forceinline__ double2 nco_cmul(double2 a, double2 b)
{
    return make_double2(__fma_rn(a.x, b.x, -__dmul_rn(a.y, b.y)), __fma_rn(a.x, b.y, __dmul_rn(a.y, b.x)));
}
__device__ __forceinline__ float2 nco_f(double2 p) { return make_float2(float(p.x), float(p.y)); }
__device__ __forceinline__ float4 nco_f4(double2 p) { const float2 f = nco_f(p); return make_float4(f.x, f.x, f.y, f.y); }
__device__ __forceinline__ float2 cmul2(float2 a, float2 b)   // packed FMUL2
{
    unsigned long long ra = *reinterpret_cast<unsigned long long*>(&a), rb = *reinterpret_cast<unsigned long long*>(&b), rd;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
    return *reinterpret_cast<float2*>(&rd);
}
__device__ __forceinline__ float2 cfma2(float2 a, float2 b, float2 c)   // packed FFMA2, per-component operands
{
    unsigned long long ra = *reinterpret_cast<unsigned long long*>(&a), rb = *reinterpret_cast<unsigned long long*>(&b),
                       rc = *reinterpret_cast<unsigned long long*>(&c), rd;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
    return *reinterpret_cast<float2*>(&rd);
}
// phasor(j) = cf32(E * S1) (x) cf32(S2):  (a + ib)(c + id) = (a, a) * (c, d) + (b, b) * (-d, c), two packed operations;
// s2r = (-d, c) is a lane constant.  One fixed operation order everywhere (FIR loop, boundary pieces, carry): the value
// depends on j only.
__device__ __forceinline__ float2 nco_phasor(float4 pq, float2 s2, float2 s2r)
{
    return cfma2(make_float2(pq.z, pq.w), s2r, cmul2(make_float2(pq.x, pq.y), s2));
}
// y = x * phasor:  (xr + i xi)(pr + i pi) = (xr, xi) * (pr, pr) + (-xi, xr) * (pi, pi)
__device__ __forceinline__ float2 nco_apply(float2 x, float2 ph)
{
    return cfma2(make_float2(-x.y, x.x), make_float2(ph.y, ph.y), cmul2(x, make_float2(ph.x, ph.x)));
}
__device__ __forceinline__ void nco_fill_e(NcoWarpSmem& ns, const NcoChan& nc, int ebase, int lane)
{
    __syncwarp();
    ns.e[lane] = nco_cis(__dadd_rn(nc.ph0, __dmul_rn(double(ebase + lane) * 4096.0, nc.inc)));
    __syncwarp();
}

// F: input format (iq_format.cuh).  An integer format streams the integers (2 or 4 B per sample instead of 8) into the ring;
// interior pieces are widened in registers on their way into the FIR, boundary pieces (carry, ragged channel ends) in
// place first -- the same values either way, so the result is bit for bit that of the cf32 kernel on the widened input.
template <int M, int T, bool NCO, int F = HBD_IQ_CF32>
__global__ void __launch_bounds__(K1Cfg<NCO>::kWarps * 32, 1)
decim1_kernel(DecimArgs a)
{
    using In = typename IqFmt<F>::T;
    constexpr bool kInt = F != HBD_IQ_CF32;
    constexpr int kG = 16 / int(sizeof(In));   // samples per 16-byte TMA granule
    static_assert(!(NCO && kInt), "the fused NCO reads cf32");
    constexpr int kWarps = K1Cfg<NCO>::kWarps;
    using G = Geo<M, T, K1Cfg<NCO>::kPsbMin>;
    using WS = WarpSmem<M, T, K1Cfg<NCO>::kPsbMin, K1Cfg<NCO>::kSt, kG>;
    constexpr int kSt = K1Cfg<NCO>::kSt;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    WS& sm = reinterpret_cast<WS*>(smem_raw)[warp];
    NcoWarpSmem& ns = reinterpret_cast<NcoWarpSmem*>(smem_raw + sizeof(WS) * kWarps)[NCO ? warp : 0];

    if (lane == 0) {
        for (int s = 0; s < kSt; ++s) mbar_init(&sm.full[s], 1);
        fence_mbar_init();
    }
    __syncwarp();

    // taps stay in registers: lane sees positions P0 = lane and P1 = lane + 32 of every superblock
    float h0[G::NLIVE], h1[G::NLIVE];
#pragma unroll
    for (int j = 0; j < G::NLIVE; ++j) {
        h0[j] = tap_for<M, T>(a.taps, j + 1, lane);
        h1[j] = tap_for<M, T>(a.taps, j + 1, lane + 32);
    }

    // streamed-once input (not the wideband capture row that every channel re-reads through its NCO)
    constexpr bool kHint = HBD_K1_EVICT_FIRST && !NCO;
    const uint64_t l2_first = kHint ? l2_policy_evict_first() : 0ull;
    uint32_t phase_bits = 0; // parity per ring slot
    // Work = the (channel, superblock) plane flattened; every warp takes ONE contiguous span of it, so the
    // ramp-in (RAMP superblocks whose outputs are discarded) is paid once per span and once per channel start
    // instead of once per 128 superblocks, and all warps finish together (no wave quantisation).
    const long long total_sb = (long long)a.n_channels * a.sb_per_channel;
    long long g = (long long)(blockIdx.x * kWarps + warp) * a.span;
    const long long g_end = g + a.span < total_sb ? g + a.span : total_sb;

    while (g < g_end) {
        const int chl = int(g / a.sb_per_channel);
        const int b_lo = int(g - (long long)chl * a.sb_per_channel);
        const int b_span_hi = int(g_end - g < (long long)(a.sb_per_channel - b_lo) ? b_lo + (g_end - g) : a.sb_per_channel);
        g += b_span_hi - b_lo;
        const int ch = a.ch0 + chl;
        const ChanPlan pl = a.uniform ? a.uplan : a.plan[ch];
        const In* chunk = reinterpret_cast<const In*>(a.chunk) + (size_t)ch * a.chunk_pitch;
        const float2* carry = a.carry + (size_t)ch * a.carry_cap + a.carry_cap; // carry[j] valid for -carry_cap <= j < 0
        auto sample = [&](int j) { return (j < 0) ? carry[j] : IqFmt<F>::dq(chunk[j]); };
        // superblock b covers step-local sample positions x in (64(b-1), 64b]; the outputs k with
        // (b-1)*NOUT < k <= b*NOUT end inside it.  This span owns superblocks [b_lo, b_hi) of the channel.
        const int n1 = int(pl.n1);
        const int n_sb_total = (n1 - 1 + G::NOUT - 1) / G::NOUT + 1;       // superblocks 0 .. ceil((n1-1)/NOUT)
        NcoChan nc{};
        bool mixing = false;
        int ebase = 0;
        if (NCO) {
            nc = a.nco[ch];
            mixing = !(nc.inc == 0.0 && nc.ph0 == 0.0);                     // a channel without an offset is a plain copy (nco.cu)
            if (mixing) {
                __syncwarp();
                for (int k = lane; k < 64; k += 32) {
                    ns.s1[k] = nco_cis(__dmul_rn(double(64 * k), nc.inc));
                    ns.s2[k] = nco_f(nco_cis(__dmul_rn(double(k), nc.inc)));
                }
                nco_fill_e(ns, nc, ebase, lane);
            }
        }
        if (!(pl.flags & 1u) && b_lo < n_sb_total) {
        const int b_hi = min(b_span_hi, n_sb_total);
        const int b_first = b_lo - G::RAMP_GROUPS * G::U;                   // ramp-in: whole groups, outputs discarded
        const int n_groups = (b_hi - b_first + G::U - 1) / G::U;
        const int n_pieces = (n_groups + G::GROUPS_PER_PIECE - 1) / G::GROUPS_PER_PIECE;
        // outputs this span may store
        const int k_lo = max(0, (b_lo - 1) * G::NOUT + 1), k_hi = min(n1, (b_hi - 1) * G::NOUT + 1);

        // sample addressing: j = x - r indexes the pushed chunk (j >= 0) or the carry (j < 0);
        // everything below is relative to the first sample of the walk, jw = j - j0 >= 0
        const int j0 = 64 * (b_first - 1) + 1 - int(pl.r);
        const int odd = j0 & (kG - 1);         // ring sample s holds j = (j0 - odd) + p*PIECE_SAMPLES + s
        const int j_cap_lo = -a.carry_cap, j_end = int(pl.n);

        // ---- producer: copy piece p into its ring slot ----------------------------------------------------
        auto issue_piece = [&](int p) {
            const int slot = p % kSt;
            unsigned char* dst = sm.ring[slot];
            const int A = j0 - odd + p * G::PIECE_SAMPLES;          // j of ring sample 0 (granule aligned)
            const int want_lo = A + odd, want_hi = want_lo + G::PIECE_SAMPLES;
            const int lo = max(A, j_cap_lo);                          // granule aligned
            const int hi = min(A + G::PIECE_SAMPLES + (kInt ? (odd ? kG : 0) : 2 * odd), j_end);
            const int hi2 = max(hi & ~(kG - 1), lo);                  // 16-byte granular end of the TMA part
            if (lane == 0) {
                if (hi2 > lo) {
                    const int c_hi = min(hi2, 0), d_lo = max(lo, 0);
                    // the slot last held generic-proxy stores (reduction rows, widened boundary samples)
                    if (WS::kRedInRing || kInt) fence_proxy_async();
                    if (kInt) mbar_expect_tx(&sm.full[slot], uint32_t(max(c_hi - lo, 0)) * 8u + uint32_t(max(hi2 - d_lo, 0)) * uint32_t(sizeof(In)));
                    else mbar_expect_tx(&sm.full[slot], uint32_t(hi2 - lo) * 8u);
                    if (c_hi > lo) tma_load_1d(dst + (lo - A) * 8, carry + lo, uint32_t(c_hi - lo) * 8u, &sm.full[slot]);
                    if (hi2 > d_lo) {
                        unsigned char* dd = kInt ? dst + WS::kIntOff + (d_lo - A) * int(sizeof(In)) : dst + (d_lo - A) * 8;
                        if (kHint) tma_load_1d_hint(dd, chunk + d_lo, uint32_t(hi2 - d_lo) * uint32_t(sizeof(In)), &sm.full[slot], l2_first);
                        else tma_load_1d(dd, chunk + d_lo, uint32_t(hi2 - d_lo) * uint32_t(sizeof(In)), &sm.full[slot]);
                    }
                } else {
                    mbar_arrive(&sm.full[slot]);
                }
            }
            if (!kInt && (lo > want_lo || hi2 < want_hi)) { // rare: TMA part does not cover the wanted range (ends of a channel)
                float2* d2 = reinterpret_cast<float2*>(dst);
                for (int j = want_lo + lane; j < want_hi; j += 32) {
                    if (j >= lo && j < hi2) continue;                 // delivered by the bulk copy
                    // odd trailing sample of an odd-length chunk: plain copy; everything not backed by data: zero
                    // (stale shared memory could hold NaN patterns and 0 * NaN would poison a valid output)
                    d2[j - A] = (j >= lo && j < hi) ? sample(j) : make_float2(0.f, 0.f);
                }
            }
        };

        // WAR note: a ring slot is only re-filled by the warp that has finished reading it
        // (program order + __syncwarp), so no "empty" barrier is needed.
        __syncwarp();
        for (int p = 0; p < min(kSt - 1, n_pieces); ++p) issue_piece(p);

        float2 acc[G::NLIVE];
#pragma unroll
        for (int j = 0; j < G::NLIVE; ++j) acc[j] = make_float2(0.f, 0.f);

        float2* out = a.s1 + (size_t)ch * a.s1_pitch + a.s1_hist;
        int k_next = (b_first - 1) * G::NOUT + 1;   // output index that completes next
        int staged = 0;                              // NOUT > 1 only: rows waiting in sm.red

        for (int p = 0; p < n_pieces; ++p) {
            const int slot = p % kSt;
            __syncwarp(); // every lane is done reading the slot that is about to be refilled
            if (p + kSt - 1 < n_pieces) issue_piece(p + kSt - 1);
            mbar_wait(&sm.full[slot], (phase_bits >> slot) & 1u);
            phase_bits ^= 1u << slot;
            __syncwarp();
            // ---- fused NCO: samples 0 <= j < n of the raw chunk get their phasor; j < 0 is the already mixed carry ----------
            // A piece that lies completely inside [0, n) (all but the first and last of a channel) is mixed in REGISTERS on
            // its way into the FIR; a boundary piece is mixed in place first.  Same phasor, same operation order either way.
            bool mix_in_loop = false;
            float2 s2a = make_float2(1.f, 0.f), s2ar = make_float2(0.f, 1.f), s2b = s2a, s2br = s2ar;
            int w0 = 0, w1 = 0;
            if (NCO && mixing) {
                const int jp = j0 + p * G::PIECE_SAMPLES;                    // j of this lane-0 sample of superblock 0
                const int j_last = min(jp + G::PIECE_SAMPLES - 1, j_end - 1);
                if (j_last >= 0) {
                    const int b_min = max(jp, 0) >> 12, b_max = j_last >> 12;
                    if (b_min < ebase || b_max >= ebase + 32) { ebase = b_min; nco_fill_e(ns, nc, ebase, lane); }
                    const int q0 = jp >> 6;                                   // floor: jp may be negative
                    __syncwarp();
                    if (lane <= G::PSB) {
                        const int q = q0 + lane;
                        if (q >= 0 && (q >> 6) < ebase + 32) ns.pq[lane] = nco_f4(nco_cmul(ns.e[(q >> 6) - ebase], ns.s1[q & 63]));
                    }
                    __syncwarp();
                    const int c0 = jp & 63;
                    w0 = (c0 + lane) >> 6; w1 = (c0 + lane + 32) >> 6;
                    s2a = ns.s2[(c0 + lane) & 63]; s2b = ns.s2[(c0 + lane + 32) & 63];
                    s2ar = make_float2(-s2a.y, s2a.x); s2br = make_float2(-s2b.y, s2b.x);
                    mix_in_loop = jp >= 0 && jp + G::PIECE_SAMPLES <= j_end;
                    if (!mix_in_loop) {
                        float2* px = reinterpret_cast<float2*>(sm.ring[slot]) + odd + lane;
#pragma unroll 1
                        for (int sb = 0; sb < G::PSB; ++sb) {
                            const int j = jp + sb * 64 + lane;
                            const float2 xa = px[sb * 64], xb = px[sb * 64 + 32];
                            const float2 ya = nco_apply(xa, nco_phasor(ns.pq[sb + w0], s2a, s2ar)), yb = nco_apply(xb, nco_phasor(ns.pq[sb + w1], s2b, s2br));
                            __syncwarp();
                            if (j >= 0 && j < j_end) px[sb * 64] = ya;
                            if (j + 32 >= 0 && j + 32 < j_end) px[sb * 64 + 32] = yb;
                        }
                        __syncwarp();
                    }
                }
            }
            // ---- integer input: a piece that the integers cover completely (all but the first and last of a channel) is widened
            // in registers on its way into the FIR; a boundary piece (carry samples, ragged ends) is widened in place first
            bool int_in_loop = false;
            if (kInt) {
                const int A = j0 - odd + p * G::PIECE_SAMPLES;    // as in issue_piece
                const int want_lo = A + odd, want_hi = want_lo + G::PIECE_SAMPLES;
                const int lo = max(A, j_cap_lo);
                const int hi = min(A + G::PIECE_SAMPLES + (odd ? kG : 0), j_end);
                const int hi2 = max(hi & ~(kG - 1), lo);
                int_in_loop = A >= 0 && hi2 >= want_hi;
                if (!int_in_loop) {
                    float2* d2 = reinterpret_cast<float2*>(sm.ring[slot]);
                    const In* q = reinterpret_cast<const In*>(sm.ring[slot] + WS::kIntOff);
                    const int s_hi = hi2 - A;
#pragma unroll 1
                    for (int s0 = max(lo, 0) - A; s0 < s_hi; s0 += 32) {   // ring positions delivered as integers, in place
                        const int s = s0 + lane;
                        float2 v = make_float2(0.f, 0.f);
                        if (s < s_hi) v = IqFmt<F>::dq(q[s]);
                        __syncwarp();
                        if (s < s_hi) d2[s] = v;
                    }
                    __syncwarp();
                    if (lo > want_lo || hi2 < want_hi) {   // what the bulk copies did not deliver, as in the cf32 kernel
                        for (int j = want_lo + lane; j < want_hi; j += 32) {
                            if (j >= lo && j < hi2) continue;
                            d2[j - A] = (j >= lo && j < hi) ? sample(j) : make_float2(0.f, 0.f);
                        }
                    }
                    __syncwarp();
                }
            }
            const float2* src = reinterpret_cast<const float2*>(sm.ring[slot]) + odd + lane;
            const In* qsrc = reinterpret_cast<const In*>(sm.ring[slot] + WS::kIntOff) + odd + lane;
            float2 (*red)[kRedPitch] = WS::kRedInRing ? reinterpret_cast<float2 (*)[kRedPitch]>(sm.ring[slot]) : sm.red;

            // the FIR over the piece; `load(i)` yields sample i of it (the branch on the input path is taken once per piece)
            auto fir_piece = [&](auto load) {
#pragma unroll 1
                for (int g = 0; g < G::GROUPS_PER_PIECE; ++g) {
#pragma unroll
                    for (int u = 0; u < G::U; ++u) {
                        float2 x0 = load((g * G::U + u) * 64);
                        float2 x1 = load((g * G::U + u) * 64 + 32);
                        if (NCO && mix_in_loop) {
                            x0 = nco_apply(x0, nco_phasor(ns.pq[g * G::U + u + w0], s2a, s2ar));
                            x1 = nco_apply(x1, nco_phasor(ns.pq[g * G::U + u + w1], s2b, s2br));
                        }
#pragma unroll
                        for (int j = 0; j < G::NLIVE; ++j) {
                            const int r = (j + u * G::NOUT) % G::NLIVE; // register holding live output j
                            // tap index of position P for live output j (0-based): t = T - M*(j+1) + P; skip the
                            // half-superblocks where no lane has a tap (compile-time)
                            const int t0 = T - M * (j + 1);
                            if (t0 + 31 >= 0 && t0 < T) acc[r] = cfma(x0, h0[j], acc[r]);
                            if (t0 + 63 >= 0 && t0 + 32 < T) acc[r] = cfma(x1, h1[j], acc[r]);
                        }
#pragma unroll
                        for (int j = 0; j < G::NOUT; ++j) {
                            const int r = (j + u * G::NOUT) % G::NLIVE;
                            if (G::NOUT == 1) {
                                if (WS::kRedInRing) __syncwarp();     // every lane has read superblock (g*U+u) of the slot
                                red[g * G::U + u][lane] = acc[r];               // row = superblock within the piece
                            } else {
                                sm.red[staged][lane] = acc[r];
                                if (++staged == 16) { reduce_rows(sm.red, 16, k_next + j - 15, k_lo, k_hi, out, lane); staged = 0; }
                            }
                            acc[r] = make_float2(0.f, 0.f);
                        }
                        if (G::NOUT > 1) k_next += G::NOUT;
                    }
                }
            };
            if (kInt && int_in_loop) fir_piece([&](int i) { return IqFmt<F>::dq(qsrc[i]); });
            else fir_piece([&](int i) { return src[i]; });
            if (G::NOUT == 1) {
                reduce_rows(red, G::PSB, k_next, k_lo, k_hi, out, lane);
                k_next += G::PSB;
            }
        }
        if (G::NOUT > 1 && staged) reduce_rows(sm.red, staged, k_next - staged, k_lo, k_hi, out, lane);
        __syncwarp();
        }
        // The span that reaches the end of a channel also writes the channel's carry for the NEXT call
        // (Decimator.h:141-143 history + Decoder.h:432-435 unconsumed remainder): the last T-1 + r' samples of
        // [carry | chunk], r' = r + n - consumed.  It goes to the other half of a ping-pong pair because spans
        // of the same channel owned by other warps may still be reading the current carry.
        if (b_span_hi == a.sb_per_channel) {
            const int keep = T - 1 + int(pl.r + pl.n - pl.consumed);       // <= carry_cap (host sized)
            float2* next = a.carry_next + (size_t)ch * a.carry_cap + a.carry_cap;
            const int jn = int(pl.n);
            if (NCO && mixing && jn > 0) {
                const int b_min = max(jn - keep, 0) >> 12, b_max = (jn - 1) >> 12;
                if (b_min < ebase || b_max >= ebase + 32) { ebase = b_min; nco_fill_e(ns, nc, ebase, lane); }
            }
            for (int i = lane; i < keep; i += 32) {
                const int j = jn - keep + i;
                float2 v = (j < 0) ? carry[j] : IqFmt<F>::dq(chunk[j]);
                if (NCO && mixing && j >= 0) { // the carry holds MIXED samples: same phasor as above
                    const float2 s2 = ns.s2[j & 63];
                    v = nco_apply(v, nco_phasor(nco_f4(nco_cmul(ns.e[(j >> 12) - ebase], ns.s1[(j >> 6) & 63])), s2, make_float2(-s2.y, s2.x)));
                }
                next[i - keep] = v;
            }
        }
    }
}

// ---- generic fallback: one thread per output.  Used for tap tables whose T/M is large
// (d_8_r_8, d_4_r_4, d_2_r_2 as FIRST stage, i.e. total factor <= 8: input rates <= 1.3 MS/s).
__global__ void decim1_generic_kernel(DecimArgs a, int M, int T)
{
    const int ch = a.ch0 + blockIdx.y;
    const ChanPlan pl = a.uniform ? a.uplan : a.plan[ch];
    if (pl.flags & 1u) return;
    const float2* chunk = a.chunk + (size_t)ch * a.chunk_pitch;
    const float2* carry = a.carry + (size_t)ch * a.carry_cap + a.carry_cap;
    float2* out = a.s1 + (size_t)ch * a.s1_pitch + a.s1_hist;
    for (unsigned k = blockIdx.x * blockDim.x + threadIdx.x; k < pl.n1; k += gridDim.x * blockDim.x) {
        const long long j_first = (long long)k * M - (T - 1) - (long long)pl.r;
        float re = 0.f, im = 0.f;
        for (int t = 0; t < T; ++t) {
            const long long j = j_first + t;
            const float2 x = (j < 0) ? carry[j] : chunk[j];
            const float h = __ldg(a.taps + t);
            re = fmaf(x.x, h, re);
            im = fmaf(x.y, h, im);
        }
        out[k] = make_float2(re, im);
    }
}

// factor 1: no decimator at all (Decoder.h:157 default) -- the "stage-1 output" is the input
__global__ void decim1_copy_kernel(DecimArgs a)
{
    const int ch = a.ch0 + blockIdx.y;
    const ChanPlan pl = a.uniform ? a.uplan : a.plan[ch];
    if (pl.flags & 1u) return;
    const float2* chunk = a.chunk + (size_t)ch * a.chunk_pitch;
    float2* out = a.s1 + (size_t)ch * a.s1_pitch + a.s1_hist;
    for (unsigned k = blockIdx.x * blockDim.x + threadIdx.x; k < pl.n1; k += gridDim.x * blockDim.x) out[k] = chunk[k];
}

// ---- stage-1 carry for the NEXT call when K1 is not the TMA kernel: last (T1-1 + r') samples of [carry | chunk] ----
__global__ void __launch_bounds__(128)
carry_kernel(const ChanPlan* __restrict__ plan, ChanPlan uplan, int uniform, const float2* __restrict__ chunk_base, size_t chunk_pitch, const float2* __restrict__ carry_base,
             float2* __restrict__ next_base, int T1, int ch0, int carry_cap)
{
    const int ch = ch0 + blockIdx.x;
    const ChanPlan pl = uniform ? uplan : plan[ch];
    const int keep = T1 - 1 + int(pl.r + pl.n - pl.consumed);             // <= carry_cap (host sized)
    const float2* carry = carry_base + (size_t)ch * carry_cap + carry_cap;
    float2* next = next_base + (size_t)ch * carry_cap + carry_cap;
    const float2* chunk = chunk_base + (size_t)ch * chunk_pitch;
    for (int i = threadIdx.x; i < keep; i += 128) {
        const long long j = (long long)pl.n - keep + i;
        next[i - keep] = (j < 0) ? carry[j] : chunk[j];
    }
}

cudaError_t launch_carry(const ChanPlan* plan, ChanPlan uplan, int uniform, const float2* chunk, size_t chunk_pitch, const float2* carry, float2* carry_next, int T1, int ch0,
                         int n_channels, int carry_cap, cudaStream_t stream, int* launches)
{
    carry_kernel<<<n_channels, 128, 0, stream>>>(plan, uplan, uniform, chunk, chunk_pitch, carry, carry_next, T1, ch0, carry_cap);
    if (launches) ++*launches;
    return cudaGetLastError();
}

constexpr int kMinSpan = 48; // superblocks: keeps the ramp-in below ~12 % when there are few channels

template <int M, int T, bool NCO = false, int F = HBD_IQ_CF32>
static cudaError_t launch_fast(DecimArgs a, unsigned max_n1, int n_sms, cudaStream_t stream, int* launches)
{
    constexpr int kWarps = K1Cfg<NCO>::kWarps;
    using G = Geo<M, T, K1Cfg<NCO>::kPsbMin>;
    const size_t smem = sizeof(WarpSmem<M, T, K1Cfg<NCO>::kPsbMin, K1Cfg<NCO>::kSt, 16 / int(sizeof(typename IqFmt<F>::T))>) * kWarps +
                        (NCO ? sizeof(NcoWarpSmem) * kWarps : 0);
    static bool configured = false; // one device per process (one process per GPU)
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(decim1_kernel<M, T, NCO, F>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        // all kernels of the path ask for the same (maximum) shared-memory carve-out so that the low-priority tail kernels
        // can co-reside with K1 on an SM instead of forcing a carve-out reconfiguration
        cudaFuncSetAttribute(decim1_kernel<M, T, NCO, F>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        configured = true;
    }
    a.sb_per_channel = max_n1 ? int((max_n1 - 1 + G::NOUT - 1) / G::NOUT + 1) : 1;
    const long long total_sb = (long long)a.n_channels * a.sb_per_channel;
    const long long warps_max = (long long)n_sms * kWarps;
    long long span = (total_sb + warps_max - 1) / warps_max;
    if (span < kMinSpan) span = kMinSpan;
    a.span = (int)span;
    const long long n_spans = (total_sb + span - 1) / span;
    int grid = (int)std::min<long long>(n_sms, (n_spans + kWarps - 1) / kWarps);
    if (grid < 1) grid = 1;
    decim1_kernel<M, T, NCO, F><<<grid, kWarps * 32, smem, stream>>>(a);
    if (launches) ++*launches;
    return cudaGetLastError();
}

cudaError_t launch_decim1(DecimArgs a, int M, int T, unsigned max_n1, int n_sms, cudaStream_t stream, int* launches, int format)
{
    if (format != HBD_IQ_CF32) {   // integer input read natively: the /64 first stage only (decim1_supports_native_iq)
        if (a.nco || !decim1_supports_native_iq(M, T)) return cudaErrorInvalidValue;
        switch (format) {
        case HBD_IQ_CS16: return launch_fast<64, 348, false, HBD_IQ_CS16>(a, max_n1, n_sms, stream, launches);
        case HBD_IQ_CS8: return launch_fast<64, 348, false, HBD_IQ_CS8>(a, max_n1, n_sms, stream, launches);
        case HBD_IQ_CU8: return launch_fast<64, 348, false, HBD_IQ_CU8>(a, max_n1, n_sms, stream, launches);
        default: return cudaErrorInvalidValue;
        }
    }
    if (a.nco) {   // fused NCO: only the /64 first stage has it (decim1_supports_fused_nco)
        if (M == 64 && T == 348) return launch_fast<64, 348, true>(a, max_n1, n_sms, stream, launches);
        return cudaErrorInvalidValue;
    }
    if (M == 64 && T == 348) return launch_fast<64, 348>(a, max_n1, n_sms, stream, launches);
    if (M == 32 && T == 174) return launch_fast<32, 174>(a, max_n1, n_sms, stream, launches);
    if (M == 32 && T == 212) return launch_fast<32, 212>(a, max_n1, n_sms, stream, launches);
    if (M == 16 && T == 107) return launch_fast<16, 107>(a, max_n1, n_sms, stream, launches);
    if (M == 8 && T == 54) return launch_fast<8, 54>(a, max_n1, n_sms, stream, launches);
    if (max_n1) {
        dim3 grid((max_n1 + 255) / 256, a.n_channels);
        if (grid.x > 1024) grid.x = 1024;
        if (M == 1) decim1_copy_kernel<<<grid, 256, 0, stream>>>(a);
        else decim1_generic_kernel<<<grid, 256, 0, stream>>>(a, M, T);
        if (launches) ++*launches;
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    return launch_carry(a.plan, a.uplan, a.uniform, a.chunk, a.chunk_pitch, a.carry, a.carry_next, T, a.ch0, a.n_channels, a.carry_cap, stream, launches);
}

bool decim1_supports_fused_nco(int M, int T) { return M == 64 && T == 348; }
bool decim1_supports_native_iq(int M, int T) { return M == 64 && T == 348; }

} // namespace hbd
