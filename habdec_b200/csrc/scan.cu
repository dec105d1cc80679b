// Wideband scanner: averaged power spectrum (Welch) of a whole capture, and the C ABI of hbd_scanner.
//
// Spectrum (include/habdec_b200.h, hbd_scan_*): segments of N samples at hop N/2, 4-term Blackman-Harris window
// (habdec_windows.h:27-53, evaluated in float64 on the host, stored as float32), |X_s[k]|^2 in float32, summed over the
// segments in float64, in segment order, one addition per segment.  Every segment is computed the same way wherever its
// samples come from (the carry of earlier pushes, a host upload, a device capture read in place), so the spectrum does
// not depend on how a capture is cut into pushes, and an integer push equals the cf32 push of its dequantised values.
//
// Four-step transform, N = 4096 * R (n = R n1 + r, k = k1 + 4096 k2):
//   X[k1 + 4096 k2] = sum_r W_R^(r k2) [ W_N^(r k1) sum_n1 w[R n1 + r] x[R n1 + r] W_4096^(n1 k1) ]
//   pass A (scan_fft_kernel): one CTA per (segment, r): fft4096 of the windowed, widened samples; the twiddle W_N^(r k1)
//          from the float64-evaluated table; out Y[s][r][k1], coalesced through the exchange area.  The window and the
//          twiddles are stored per r ([r][n1], [r][k1]), so that a CTA reads both as contiguous rows.
//   pass B (scan_accum_kernel): one CTA per 16 columns k1: for each segment in order the R-point DFT over r (radix 2 in
//          shared memory), |X|^2, and the float64 sums of its 16 R bins kept in registers across the batch.
// A batch holds at most 2^22 / N segments, so Y (32 MB) stays in L2 between the two passes.  No cuFFT.
#include "../../include/habdec_b200.h"
#include "cuda_res.h"
#include "fft_dev.cuh"
#include "iq_format.cuh"
#include "scan.cuh"

#include <cmath>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <vector>

namespace hbd {

template <int F>
__device__ __forceinline__ float2 scan_sample(const ScanSrc& s, size_t q)
{
    using T = typename IqFmt<F>::T;
    return q < s.m ? s.carry[q] : IqFmt<F>::dq(static_cast<const T*>(s.src)[q - s.m]);
}

// grid (R, n_seg), 256 threads
template <int F>
__global__ void __launch_bounds__(kFftThreads)
scan_fft_kernel(ScanSrc s, size_t first, int N, const float* __restrict__ win, const float2* __restrict__ tw, float2* __restrict__ inter)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* s_a = reinterpret_cast<float2*>(smem_raw);
    const int r = blockIdx.x, R = gridDim.x, t = threadIdx.x;
    const size_t s0 = first + size_t(blockIdx.y) * size_t(N / 2);
    // windowing is an explicit unfused multiply, so every input format reaches the transform with the same values
    const float* __restrict__ w_r = win + size_t(r) * 4096;   // w[R n1 + r]
    auto load = [&](int n1) {
        const float2 x = scan_sample<F>(s, s0 + size_t(R * n1 + r));
        const float w = w_r[n1];
        return make_float2(__fmul_rn(w, x.x), __fmul_rn(w, x.y));
    };
    fft4096_load(load, tw + N, tw + N + 4096, s_a, [&](int, int k, float2 z) { s_a[k + (k >> 4)] = z; });
    __syncthreads();
    float2* out = inter + (size_t(blockIdx.y) * size_t(R) + size_t(r)) * 4096;
#pragma unroll
    for (int m = 0; m < 16; ++m) {
        const int k = t + 256 * m;
        float2 z = s_a[k + (k >> 4)];
        if (r) z = cmul(z, tw[r * 4096 + k]);      // W_N^(r k1), table [r][k1]
        out[k] = z;
    }
}

// grid 256 CTAs (16 of the 4096 columns k1 each), 256 threads; R = 2^logR rows
__global__ void __launch_bounds__(256, 2)
scan_accum_kernel(const float2* __restrict__ inter, int n_seg, int logR, const float2* __restrict__ tw_R, double* __restrict__ acc)
{
    __shared__ float2 s[16 * 257];           // [column][row], row pitch R + 1
    const int R = 1 << logR, P = R + 1, t = threadIdx.x, c0 = blockIdx.x * 16;
    const int n_el = 16 * R;                 // elements of the tile: e = 16 row + column
    double sum[16];
#pragma unroll
    for (int q = 0; q < 16; ++q) {
        const int e = t + 256 * q;
        sum[q] = e < n_el ? acc[c0 + (e & 15) + 4096 * (e >> 4)] : 0.0;
    }
    for (int b = 0; b < n_seg; ++b) {
        const float2* y = inter + size_t(b) * size_t(R) * 4096;
        __syncthreads();                     // the previous segment's tile has been read
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            const int e = t + 256 * q;
            if (e < n_el) {
                const int row = e >> 4, col = e & 15;
                const int rr = logR ? int(__brev(unsigned(row)) >> (32 - logR)) : 0;
                s[col * P + rr] = y[size_t(row) * 4096 + c0 + col];
            }
        }
        __syncthreads();
        // radix-2 DIT over the rows, bit-reversed in, natural order out; W_(2h)^p = W_R^(p R / 2h)
        for (int h = 1; h < R; h <<= 1) {
            const int tw_step = R / (2 * h);
            for (int u = t; u < 8 * R; u += 256) {
                const int col = u & 15, j = u >> 4;
                const int p = j & (h - 1), i0 = (j - p) * 2 + p;
                float2* x = s + col * P;
                const float2 a = x[i0], v = cmul(x[i0 + h], tw_R[p * tw_step]);
                x[i0] = cadd(a, v);
                x[i0 + h] = csub(a, v);
            }
            __syncthreads();
        }
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            const int e = t + 256 * q;
            if (e < n_el) {
                const float2 z = s[(e & 15) * P + (e >> 4)];
                sum[q] += double(__fadd_rn(__fmul_rn(z.x, z.x), __fmul_rn(z.y, z.y)));
            }
        }
    }
#pragma unroll
    for (int q = 0; q < 16; ++q) {
        const int e = t + 256 * q;
        if (e < n_el) acc[c0 + (e & 15) + 4096 * (e >> 4)] = sum[q];
    }
}

template <int F>
__global__ void scan_carry_kernel(ScanSrc s, size_t start, size_t count, float2* __restrict__ dst)
{
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < count; i += size_t(gridDim.x) * blockDim.x)
        dst[i] = scan_sample<F>(s, start + i);
}

constexpr size_t kScanSmem = size_t(16 * 16 * 17) * sizeof(float2);   // fft4096's exchange area, 34 KB

template <int F>
static cudaError_t launch_fft(const ScanSrc& s, size_t first, int n_seg, int N, const float* win, const float2* tw, float2* inter,
                              cudaStream_t stream)
{
    scan_fft_kernel<F><<<dim3(unsigned(N / 4096), unsigned(n_seg)), kFftThreads, kScanSmem, stream>>>(s, first, N, win, tw, inter);
    return cudaGetLastError();
}

cudaError_t launch_scan_segments(const ScanSrc& s, size_t first, int n_seg, int N, const float* win, const float2* tw, float2* inter,
                                 double* acc, cudaStream_t stream)
{
    if (n_seg <= 0) return cudaSuccess;
    cudaError_t e;
    switch (s.format) {
    case HBD_IQ_CF32: e = launch_fft<HBD_IQ_CF32>(s, first, n_seg, N, win, tw, inter, stream); break;
    case HBD_IQ_CS16: e = launch_fft<HBD_IQ_CS16>(s, first, n_seg, N, win, tw, inter, stream); break;
    case HBD_IQ_CS8: e = launch_fft<HBD_IQ_CS8>(s, first, n_seg, N, win, tw, inter, stream); break;
    case HBD_IQ_CU8: e = launch_fft<HBD_IQ_CU8>(s, first, n_seg, N, win, tw, inter, stream); break;
    default: return cudaErrorInvalidValue;
    }
    if (e != cudaSuccess) return e;
    int logR = 0;
    while ((4096 << logR) < N) ++logR;
    scan_accum_kernel<<<256, 256, 0, stream>>>(inter, n_seg, logR, tw + N + 4096 + 256, acc);
    return cudaGetLastError();
}

cudaError_t launch_scan_carry(const ScanSrc& s, size_t start, size_t count, float2* dst, cudaStream_t stream)
{
    if (!count) return cudaSuccess;
    const unsigned grid = unsigned(std::min<size_t>((count + 255) / 256, 1024));
    switch (s.format) {
    case HBD_IQ_CF32: scan_carry_kernel<HBD_IQ_CF32><<<grid, 256, 0, stream>>>(s, start, count, dst); break;
    case HBD_IQ_CS16: scan_carry_kernel<HBD_IQ_CS16><<<grid, 256, 0, stream>>>(s, start, count, dst); break;
    case HBD_IQ_CS8: scan_carry_kernel<HBD_IQ_CS8><<<grid, 256, 0, stream>>>(s, start, count, dst); break;
    case HBD_IQ_CU8: scan_carry_kernel<HBD_IQ_CU8><<<grid, 256, 0, stream>>>(s, start, count, dst); break;
    default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

} // namespace hbd

using namespace hbd;

struct hbd_scanner {
    std::mutex mtx;
    std::string err;
    int device = 0;
    int N = 0;
    int max_batch = 1;                 // segments per launch pair: 2^22 / N, Y = 32 MB
    cudaStream_t stream = nullptr;
    Stream own_stream;                 // declared before the buffers and events, so it is destroyed after them
    Event ev_up;                       // a host push's upload has been read
    DevPtr<float> d_win;
    DevPtr<float2> d_tw, d_inter;
    DevPtr<double> d_acc;
    DevPtr<float2> d_carry[2];
    int cur = 0;                       // d_carry[cur] holds the m samples from the next segment's start on
    size_t m = 0;
    Rows<unsigned char> up;            // host push staging, one row of `pitch` bytes
    double fs = 0;
    bool fs_set = false;
    unsigned long long n_seg = 0;
    double win_sq = 0;                 // sum of the (float32) window values squared, in float64

    int fail(int rc, const std::string& what) { err = what; return rc; }
    int cuda_fail(cudaError_t e, const char* what) { return fail(HBD_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e)); }
    int process(const void* src, int format, size_t n);
    ~hbd_scanner() { cudaSetDevice(device); if (stream) cudaStreamSynchronize(stream); }   // then the members release themselves
};

// the capture's next n samples (device memory, `format`) after the carry: every segment that is complete now, then the new carry
int hbd_scanner::process(const void* src, int format, size_t n)
{
    const size_t H = size_t(N / 2), total = m + n;
    const size_t S = total >= size_t(N) ? (total - size_t(N)) / H + 1 : 0;
    const ScanSrc s{d_carry[cur].get(), m, src, format};
    for (size_t b = 0; b < S; b += size_t(max_batch)) {
        const int nb = int(std::min<size_t>(size_t(max_batch), S - b));
        const cudaError_t e = launch_scan_segments(s, b * H, nb, N, d_win.get(), d_tw.get(), d_inter.get(), d_acc.get(), stream);
        if (e != cudaSuccess) return cuda_fail(e, "scan kernels");
    }
    const size_t next = S * H, keep = total - next;   // < N
    if (!S) {   // no segment completed: the new samples are appended to the carry in place (most pushes at large N)
        const cudaError_t e = launch_scan_carry(s, m, n, d_carry[cur].get() + m, stream);
        if (e != cudaSuccess) return cuda_fail(e, "scan carry");
    } else {
        const cudaError_t e = launch_scan_carry(s, next, keep, d_carry[cur ^ 1].get(), stream);
        if (e != cudaSuccess) return cuda_fail(e, "scan carry");
        cur ^= 1;
    }
    m = keep;
    n_seg += S;
    return HBD_OK;
}

extern "C" {

int hbd_scanner_create(int cuda_device, size_t n_fft, hbd_scanner** out)
{
    if (!out) return HBD_ERR_ARG;
    *out = nullptr;
    if (n_fft < size_t(kScanNMin) || n_fft > size_t(kScanNMax) || (n_fft & (n_fft - 1))) return HBD_ERR_ARG;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || cuda_device < 0 || cuda_device >= count) return HBD_ERR_CUDA;
    if (cudaSetDevice(cuda_device) != cudaSuccess) return HBD_ERR_CUDA;
    std::unique_ptr<hbd_scanner> s(new (std::nothrow) hbd_scanner);
    if (!s) return HBD_ERR_NOMEM;
    const size_t N = n_fft;
    s->device = cuda_device;
    s->N = int(N);
    s->max_batch = int(std::max<size_t>(1, (size_t(1) << 22) / N));
    if (stream_create(s->own_stream) != cudaSuccess) return HBD_ERR_CUDA;
    s->stream = s->own_stream.get();
    if (event_create(s->ev_up) != cudaSuccess) return HBD_ERR_CUDA;
    if (dev_alloc(s->d_win, N) != cudaSuccess || dev_alloc(s->d_tw, N + 4096 + 256 + N / 4096) != cudaSuccess ||
        dev_alloc(s->d_inter, size_t(s->max_batch) * N) != cudaSuccess || dev_alloc(s->d_acc, N) != cudaSuccess ||
        dev_alloc(s->d_carry[0], N) != cudaSuccess || dev_alloc(s->d_carry[1], N) != cudaSuccess) return HBD_ERR_NOMEM;
    // 4-term Blackman-Harris (habdec_windows.h:27-53), float64 -> float32, stored [r][n1] = w[R n1 + r]
    const size_t R = N / 4096;
    std::vector<float> w(N);
    const double a0 = 0.35874, a1 = 0.48829, a2 = 0.14128, a3 = 0.01168, den = double(N - 1);
    for (size_t i = 0; i < N; ++i) {
        const double x = double(i);
        const float wi = float(a0 - a1 * std::cos(2.0 * M_PI * x / den) + a2 * std::cos(4.0 * M_PI * x / den) - a3 * std::cos(6.0 * M_PI * x / den));
        w[(i % R) * 4096 + i / R] = wi;
        s->win_sq += double(wi) * double(wi);
    }
    // [r][k1] = W_N^(r k1) (N entries); the pass-1 [k1][t] and pass-2 [j1][m2] twiddles of fft4096 (as hbd_decoder::alloc_fft);
    // W_R^j (R entries).  All exp(-2 pi i num / den) evaluated in float64.
    std::vector<float2> tw(N + 4096 + 256 + R);
    auto cw = [](double num, double den) { const double ang = -2.0 * M_PI * num / den; return make_float2(float(std::cos(ang)), float(std::sin(ang))); };
    for (size_t r = 0; r < R; ++r) for (size_t k1 = 0; k1 < 4096; ++k1) tw[r * 4096 + k1] = cw(double(r * k1), double(N));
    for (size_t k1 = 0; k1 < 16; ++k1) for (size_t t = 0; t < 256; ++t) tw[N + k1 * 256 + t] = cw(double(t * k1), 4096.0);
    for (size_t j1 = 0; j1 < 16; ++j1) for (size_t m2 = 0; m2 < 16; ++m2) tw[N + 4096 + j1 * 16 + m2] = cw(double(16 * m2 * j1), 4096.0);
    for (size_t j = 0; j < R; ++j) tw[N + 4096 + 256 + j] = cw(double(j), double(R));
    if (cudaMemcpy(s->d_win.get(), w.data(), N * sizeof(float), cudaMemcpyHostToDevice) != cudaSuccess ||
        cudaMemcpy(s->d_tw.get(), tw.data(), tw.size() * sizeof(float2), cudaMemcpyHostToDevice) != cudaSuccess ||
        cudaMemset(s->d_acc.get(), 0, N * sizeof(double)) != cudaSuccess) return HBD_ERR_CUDA;
    *out = s.release();
    return HBD_OK;
}

void hbd_scanner_destroy(hbd_scanner* s) { delete s; }

const char* hbd_scanner_last_error(hbd_scanner* s) { return s ? s->err.c_str() : "null handle"; }

int hbd_scanner_set_stream(hbd_scanner* s, void* cuda_stream)
{
    if (!s) return HBD_ERR_ARG;
    std::lock_guard<std::mutex> l(s->mtx);
    cudaSetDevice(s->device);
    cudaStreamSynchronize(s->stream);
    s->own_stream.reset();
    s->stream = (cudaStream_t)cuda_stream;
    return HBD_OK;
}

static int scan_push(hbd_scanner* s, const void* iq, int format, size_t n, double fs, bool device)
{
    if (!s) return HBD_ERR_ARG;
    const size_t bytes = size_t(iq_bytes(format));
    std::lock_guard<std::mutex> l(s->mtx);
    if (!bytes) return s->fail(HBD_ERR_ARG, "unknown sample format");
    if (!iq && n) return s->fail(HBD_ERR_ARG, "null sample pointer");
    if (device && (reinterpret_cast<uintptr_t>(iq) & 15)) return s->fail(HBD_ERR_ARG, "device capture must be 16-byte aligned");
    if (!(fs > 0)) return s->fail(HBD_ERR_ARG, "sampling rate must be positive");
    if (s->fs_set && fs != s->fs) return s->fail(HBD_ERR_STATE, "sampling rate differs from the latched one: hbd_scan_reset first");
    s->fs = fs; s->fs_set = true;
    if (!n) return HBD_OK;
    if (cudaSetDevice(s->device) != cudaSuccess) return s->fail(HBD_ERR_CUDA, "cudaSetDevice");
    if (device) return s->process(iq, format, n);
    // host capture: uploaded in pieces of at most 2^24 samples (the spectrum does not depend on the cut), the caller owns
    // `iq` again on return
    const size_t piece = size_t(1) << 24;
    if (s->up.grow(std::min(n, piece) * bytes, 1, 0, s->stream) != cudaSuccess) return s->fail(HBD_ERR_NOMEM, "scan upload buffer");
    for (size_t o = 0; o < n; o += piece) {
        const size_t k = std::min(piece, n - o);
        cudaError_t e = cudaMemcpyAsync(s->up.get(), static_cast<const unsigned char*>(iq) + o * bytes, k * bytes, cudaMemcpyHostToDevice, s->stream);
        if (e != cudaSuccess) return s->cuda_fail(e, "scan upload");
        const int rc = s->process(s->up.get(), format, k);
        if (rc) return rc;
        e = cudaEventRecord(s->ev_up.get(), s->stream);
        if (e == cudaSuccess) e = cudaEventSynchronize(s->ev_up.get());
        if (e != cudaSuccess) return s->cuda_fail(e, "scan upload sync");
    }
    return HBD_OK;
}

int hbd_scan_push(hbd_scanner* s, const void* iq, int format, size_t n, double fs) { return scan_push(s, iq, format, n, fs, false); }
int hbd_scan_push_device(hbd_scanner* s, const void* d_iq, int format, size_t n, double fs) { return scan_push(s, d_iq, format, n, fs, true); }

int hbd_scan_reset(hbd_scanner* s)
{
    if (!s) return HBD_ERR_ARG;
    std::lock_guard<std::mutex> l(s->mtx);
    if (cudaSetDevice(s->device) != cudaSuccess) return s->fail(HBD_ERR_CUDA, "cudaSetDevice");
    const cudaError_t e = cudaMemsetAsync(s->d_acc.get(), 0, size_t(s->N) * sizeof(double), s->stream);
    if (e != cudaSuccess) return s->cuda_fail(e, "scan reset");
    s->m = 0; s->n_seg = 0; s->fs = 0; s->fs_set = false;
    return HBD_OK;
}

// the PSD as float32, fft-shifted, into psd[N] (host); 0 while no segment is complete
static int scan_psd(hbd_scanner* s, std::vector<float>& psd)
{
    const size_t N = size_t(s->N);
    psd.assign(N, 0.0f);
    if (!s->n_seg) return HBD_OK;
    std::vector<double> acc(N);
    if (cudaSetDevice(s->device) != cudaSuccess) return s->fail(HBD_ERR_CUDA, "cudaSetDevice");
    cudaError_t e = cudaMemcpyAsync(acc.data(), s->d_acc.get(), N * sizeof(double), cudaMemcpyDeviceToHost, s->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s->stream);
    if (e != cudaSuccess) return s->cuda_fail(e, "scan read-back");
    const double den = double(s->n_seg) * s->win_sq;
    for (size_t i = 0; i < N; ++i) psd[i] = float(acc[(i + N / 2) & (N - 1)] / den);
    return HBD_OK;
}

size_t hbd_scan_get_psd(hbd_scanner* s, float* out, size_t cap_floats, unsigned long long* n_segments)
{
    if (!s) return 0;
    std::lock_guard<std::mutex> l(s->mtx);
    if (n_segments) *n_segments = s->n_seg;
    if (!out || !cap_floats) return size_t(s->N);
    std::vector<float> psd;
    if (scan_psd(s, psd)) return 0;
    memcpy(out, psd.data(), std::min(cap_floats, psd.size()) * sizeof(float));
    return size_t(s->N);
}

int hbd_scan_find(hbd_scanner* s, const hbd_scan_params* p, hbd_scan_signal* out, size_t cap)
{
    if (!s) return HBD_ERR_ARG;
    std::lock_guard<std::mutex> l(s->mtx);
    if (!s->n_seg) return 0;
    std::vector<float> psd;
    const int rc = scan_psd(s, psd);
    if (rc) return rc;
    return hbd_scan_detect(psd.data(), psd.size(), s->fs, p, out, cap);
}

} // extern "C"
