// Wideband scanner kernels (see scan.cu): averaged power spectrum of a capture, N = 4096 * R points, R = 1 .. 256.
#pragma once
#include "hbd_common.cuh"

namespace hbd {

constexpr int kScanNMin = 4096, kScanNMax = 1 << 20;

// The samples a launch reads form one virtual stream: carry[0, m) (cf32, the samples kept from earlier pushes) followed by
// src[0, n) in `format` (read in place, widened as it is loaded).
struct ScanSrc {
    const float2* carry;
    size_t m;
    const void* src;
    int format;
};

// n_seg segments of N samples starting at virtual positions first + s * N / 2: windowed N-point transform, |X|^2 in float32,
// added to acc[k] (float64, natural bin order) one segment after the other.  inter: n_seg * N cf32 of scratch.
// win: N float32 as [r][n1] = w[R n1 + r]; tw: [r][k1] = W_N^(r k1) (N entries), fft4096's pass-1 / pass-2 tables (4096 + 256,
// laid out like K4's, hbd_decoder::alloc_fft), W_R^j (R entries).
cudaError_t launch_scan_segments(const ScanSrc& s, size_t first, int n_seg, int N, const float* win, const float2* tw, float2* inter,
                                 double* acc, cudaStream_t stream);
// dst[i] = virtual[start + i], i < count (cf32)
cudaError_t launch_scan_carry(const ScanSrc& s, size_t start, size_t count, float2* dst, cudaStream_t stream);

} // namespace hbd
