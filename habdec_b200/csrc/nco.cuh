// K0 launch interface (see nco.cu): per-channel NCO pre-mixer / wideband channeliser front-end
#pragma once
#include "hbd_common.cuh"

namespace hbd {

// per channel and per push: phase in cycles of the first sample, phase increment per sample, and the rotation
// over kNcoThreads samples (all evaluated in float64 on the host)
struct NcoChan {
    double ph0;        // in [0, 1)
    double inc;        // f_nco / fs  (cycles per sample)
    double step_re, step_im; // exp(-2 pi i inc kNcoThreads)
};
constexpr int kNcoThreads = 128;
constexpr int kNcoPerThread = 8;

// dst[ch][dst_off + i] = dq(src[ch * src_pitch + i]) * exp(-2 pi i (ph0 + i inc)),  i in [0, n)
// src holds samples of `format` (HBD_IQ_*, dq = its dequantisation; src_pitch in samples).  nco == nullptr: no mixing
// (widen only).  src_pitch == 0: every channel reads the same (wideband) row.  A cf32 src may equal dst (in-place).
cudaError_t launch_nco_mix(const void* src, size_t src_pitch, float2* dst, size_t dst_pitch, size_t dst_off, size_t n,
                           const NcoChan* nco, int ch0, int n_channels, cudaStream_t stream, int* launches, int format = 0);

} // namespace hbd
