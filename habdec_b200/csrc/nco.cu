// K0 -- per-channel NCO pre-mixer (frequency-offset channels of one wideband capture, AFC retune).
//
// The reference Decoder has no mixer: its AFC only MEASURES the offset and the caller retunes the SDR
// (code/websocketServer/main.cpp:247-265), and a signal decodes only if its two tones straddle DC
// (SymbolExtractor.h:149,182,196).  For a batch of frequency-offset channels cut from one capture the retune
// becomes a per-channel complex mix in front of the decimator:
//
//     y[i] = x[i] * exp(-2 pi i * phase(i)),   phase(i) = frac(ph0 + i * f_nco / fs)
//
// phase in float64 (it must stay coherent over billions of samples), the phasor rounded to cf32, the product
// formed like std::complex<float>::operator* without FMA contraction -- the same arithmetic as the oracle
// (oracle/pyoracle.py: premix), "CPU pre-mix, then the reference Decoder" (SURVEY.md D4).
//
// Cost control: a thread evaluates ONE float64 sincospi (its first sample) and walks 8 samples spaced
// kNcoThreads apart with a float64 rotation by the host-evaluated exp(-2 pi i inc kNcoThreads); loads and stores
// are fully coalesced.  The kernel is HBM bound (8 B read + 8 B write per sample; the wideband row stays in L2).
//
// It also widens integer input (CS16 / CS8 / CU8) to cf32 for every path the decimator does not read natively: host
// pushes (uploaded as integers), wideband rows and device pushes outside K1's native case.  nco == nullptr: widen only.
#include "nco.cuh"
#include "iq_format.cuh"
#include <algorithm>

namespace hbd {

// F: input sample format (iq_format.cuh).  Integer input is widened to cf32 on the way (nco == nullptr: widen only).
template <int F>
__global__ void __launch_bounds__(kNcoThreads)
nco_mix_kernel(const typename IqFmt<F>::T* __restrict__ src, size_t src_pitch, float2* dst, size_t dst_pitch, size_t dst_off, size_t n,
               const NcoChan* __restrict__ nco, int ch0)
{
    const int ch = ch0 + blockIdx.y;
    const NcoChan c = nco ? nco[ch] : NcoChan{};
    const typename IqFmt<F>::T* s = src + size_t(ch) * src_pitch;
    float2* d = dst + size_t(ch) * dst_pitch + dst_off;
    const size_t tile = size_t(kNcoThreads) * kNcoPerThread;
    for (size_t base = size_t(blockIdx.x) * tile; base < n; base += size_t(gridDim.x) * tile) {
        const size_t i0 = base + threadIdx.x;
        if (c.inc == 0.0 && c.ph0 == 0.0) { // channel without an offset: plain copy
            if (F != HBD_IQ_CF32 || reinterpret_cast<const void*>(s) != d) {
#pragma unroll
                for (int u = 0; u < kNcoPerThread; ++u) { const size_t i = i0 + size_t(u) * kNcoThreads; if (i < n) d[i] = IqFmt<F>::dq(s[i]); }
            }
            continue;
        }
        double ph = __dadd_rn(c.ph0, __dmul_rn(double(i0), c.inc));
        ph -= floor(ph);
        double sn, cs;
        sincospi(-2.0 * ph, &sn, &cs);
#pragma unroll
        for (int u = 0; u < kNcoPerThread; ++u) {
            const size_t i = i0 + size_t(u) * kNcoThreads;
            if (i < n) {
                const float2 x = IqFmt<F>::dq(s[i]);
                const float pr = float(cs), pi = float(sn);
                float2 y;
                y.x = __fsub_rn(__fmul_rn(x.x, pr), __fmul_rn(x.y, pi));
                y.y = __fadd_rn(__fmul_rn(x.x, pi), __fmul_rn(x.y, pr));
                d[i] = y;
            }
            const double c2 = cs * c.step_re - sn * c.step_im, s2 = cs * c.step_im + sn * c.step_re;
            cs = c2; sn = s2;
        }
    }
}

template <int F>
static void launch_one(dim3 grid, cudaStream_t stream, const void* src, size_t src_pitch, float2* dst, size_t dst_pitch, size_t dst_off, size_t n,
                       const NcoChan* nco, int ch0)
{
    nco_mix_kernel<F><<<grid, kNcoThreads, 0, stream>>>(static_cast<const typename IqFmt<F>::T*>(src), src_pitch, dst, dst_pitch, dst_off, n, nco, ch0);
}

cudaError_t launch_nco_mix(const void* src, size_t src_pitch, float2* dst, size_t dst_pitch, size_t dst_off, size_t n,
                           const NcoChan* nco, int ch0, int n_channels, cudaStream_t stream, int* launches, int format)
{
    if (!iq_bytes(format)) return cudaErrorInvalidValue;
    if (!n || n_channels <= 0) return cudaSuccess;
    const size_t tile = size_t(kNcoThreads) * kNcoPerThread;
    size_t gx = (n + tile - 1) / tile;
    if (gx > 4096) gx = 4096;
    for (int c = 0; c < n_channels; c += 65535) {
        dim3 grid((unsigned)gx, (unsigned)std::min(65535, n_channels - c));
        switch (format) {
        case HBD_IQ_CF32: launch_one<HBD_IQ_CF32>(grid, stream, src, src_pitch, dst, dst_pitch, dst_off, n, nco, ch0 + c); break;
        case HBD_IQ_CS16: launch_one<HBD_IQ_CS16>(grid, stream, src, src_pitch, dst, dst_pitch, dst_off, n, nco, ch0 + c); break;
        case HBD_IQ_CS8: launch_one<HBD_IQ_CS8>(grid, stream, src, src_pitch, dst, dst_pitch, dst_off, n, nco, ch0 + c); break;
        default: launch_one<HBD_IQ_CU8>(grid, stream, src, src_pitch, dst, dst_pitch, dst_off, n, nco, ch0 + c); break;
        }
        if (launches) ++*launches;
    }
    return cudaGetLastError();
}

} // namespace hbd
