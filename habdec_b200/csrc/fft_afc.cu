// K4 -- spectrum FFT + AFC, a small grid of CTAs each owning a strided set of channels.
//
//   FFT::operator() + swap_half     code/Decoder/FFT.cpp:77-99   (FFTW3f forward c2c, unnormalised, no window)
//   FftPower / ComputeVariance / FindPeaks   code/Decoder/AFC.h:225-329
//   AFC<float>::process state machine        code/Decoder/AFC.h:92-184, Average.h:34-70
//
// FFT: 4096 = 16 x 16 x 16, fft4096 of fft_dev.cuh.  Twiddles come from a
// table evaluated in float64 on the host, so the result stays within ~1e-7 relative of a
// float64 DFT (the reference's FFTW is not in the image: parity at this boundary is
// judged against float64, SURVEY.md section 8c).  No cuFFT.
//
// AFC: the reference re-runs FftPower/FindPeaks on the same stale spectrum on every call;
// those results are cached per spectrum and only the per-call state machine (four moving
// averages, detection, stability, correction) is stepped, in float64 with explicitly
// unfused multiplies/adds so that it matches the CPU's arithmetic.
#include "hbd_common.cuh"
#include "fft_afc.cuh"
#include "fft_dev.cuh"
#include "afc_dev.cuh"
#include <algorithm>

namespace hbd {

template <typename T>
__device__ __forceinline__ T warp_sum(T v)
{
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ double block_sum(double v, double* scratch)
{
    v = warp_sum(v);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) scratch[w] = v;
    __syncthreads();
    double t = (threadIdx.x < kFftThreads / 32) ? scratch[threadIdx.x] : 0.0;
    if (w == 0) { t = warp_sum(t); if (l == 0) scratch[0] = t; }
    __syncthreads();
    return scratch[0];
}

// arg-max with first-index tie break over (value, index) pairs held one per thread
__device__ void block_argmax(float v, int i, float* sv, int* si, float& ov, int& oi)
{
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        const float ov2 = __shfl_xor_sync(0xffffffffu, v, o);
        const int oi2 = __shfl_xor_sync(0xffffffffu, i, o);
        if (ov2 > v || (ov2 == v && oi2 < i)) { v = ov2; i = oi2; }
    }
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) { sv[w] = v; si[w] = i; }
    __syncthreads();
    if (threadIdx.x == 0) {
        float bv = sv[0]; int bi = si[0];
        for (int k = 1; k < kFftThreads / 32; ++k)
            if (sv[k] > bv || (sv[k] == bv && si[k] < bi)) { bv = sv[k]; bi = si[k]; }
        sv[0] = bv; si[0] = bi;
    }
    __syncthreads();
    ov = sv[0]; oi = si[0];
}

// (sum, arg-max with first-index tie break) over one (double, float, int) triple per thread: one shuffle tree, two
// barriers; every thread folds the eight warp results itself.  `slot` selects one of two scratch sets so that two
// reductions in a row need no barrier in between.
struct RedScratch { double s[2][kFftThreads / 32]; float v[2][kFftThreads / 32]; int i[2][kFftThreads / 32]; };
__device__ __forceinline__ void block_sum_argmax(double& s, float& v, int& i, RedScratch& r, int slot)
{
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        const float ov = __shfl_xor_sync(0xffffffffu, v, o);
        const int oi = __shfl_xor_sync(0xffffffffu, i, o);
        if (ov > v || (ov == v && oi < i)) { v = ov; i = oi; }
    }
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) { r.s[slot][w] = s; r.v[slot][w] = v; r.i[slot][w] = i; }
    __syncthreads();
    s = r.s[slot][0]; v = r.v[slot][0]; i = r.i[slot][0];
#pragma unroll
    for (int k = 1; k < kFftThreads / 32; ++k) {
        s += r.s[slot][k];
        const float ov = r.v[slot][k]; const int oi = r.i[slot][k];
        if (ov > v || (ov == v && oi < i)) { v = ov; i = oi; }
    }
}

// N = 4096, the reference's size and the one on the decode path: the bins are transposed through the exchange area so
// that spectrum and power leave as coalesced rows, a thread keeps the dB values of its 16 bins in registers to the end
// (no power-spectrum staging in shared memory, no re-read), the
// statistics take two fused block reductions, the channel's state is staged in shared memory while the transform runs
// and the per-call AFC step is done by thread 0 on that copy while the other warps already load the next channel.
__global__ void __launch_bounds__(kFftThreads, 3)
fft_afc4096_kernel(FftArgs a)
{
    constexpr int N = 4096;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* s_a = reinterpret_cast<float2*>(smem_raw);
    __shared__ unsigned char s_todo[kFftThreads];
    __shared__ RedScratch s_red;
    __shared__ ChanState s_cs;
    const int t = threadIdx.x;
    {   // phase A: one thread per owned channel (see fft_afc_kernel below)
        const int j_ch = int(blockIdx.x) + t * int(gridDim.x);
        unsigned char todo = 0;
        if (j_ch < a.n_channels) {
            ChanState& sj = a.state[a.ch0 + j_ch];
            if (sj.fft_ready) todo = 1;
            else if (sj.afc_tick) { afc_step(sj, a.fs_dec, N); sj.afc_tick = 0; }
        }
        s_todo[t] = todo;
    }
    __syncthreads();
    const double inv_fs = 1.0 / a.fs_dec;
    const float2* __restrict__ tw = a.twiddle;
    for (int j = 0; int(blockIdx.x) + j * int(gridDim.x) < a.n_channels; ++j) {
        if (!s_todo[j]) continue;
        const int ch = a.ch0 + int(blockIdx.x) + j * int(gridDim.x);
        ChanState& st = a.state[ch];
        if (t < 32) {   // stage the channel's state (thread 0 steps the AFC on it at the end); warp 0 only, after its previous use
            __syncwarp();
            const unsigned* src = reinterpret_cast<const unsigned*>(&st);
            unsigned* dst = reinterpret_cast<unsigned*>(&s_cs);
            for (int i = t; i < int(sizeof(ChanState) / 4); i += 32) dst[i] = src[i];
        }
        const float2* x = a.fftbuf + (size_t)ch * N;
        float2* spec = a.spectrum + (size_t)ch * N;
        float* pw = a.power + (size_t)ch * N;
        float pdb[16];
        int bad = 0;
        // the last pass leaves bin k = kb + 256*j2 with thread kb's transpose: hand the bins over through the (now free)
        // exchange area, one pad slot per 16, so that spectrum and power go out as coalesced rows
        fft4096(x, 1, 0, tw + N, tw + N + 4096, s_a, [&](int, int k, float2 z) { s_a[k + (k >> 4)] = z; });
        __syncthreads();
#pragma unroll
        for (int m = 0; m < 16; ++m) {
            // spectrum out with the halves swapped (FFT.cpp:77-87); FftPower of the bin (AFC.h:236-286)
            const int i = t + 256 * m, k = (i + N / 2) & (N - 1);
            const float2 z = s_a[k + (k >> 4)];
            spec[i] = z;
            if (z.x != z.x || z.y != z.y || isinf(z.x) || isinf(z.y)) bad = 1;
            float p = __fadd_rn(__fmul_rn(z.x, z.x), __fmul_rn(z.y, z.y)) / float(N);
            p = __fmul_rn(p, p);
            {   // float(double(p) / fs_dec): reciprocal + one residual step (see fft_afc_kernel)
                const double xd = double(p);
                double q = xd * inv_fs;
                const double r = fma(-q, a.fs_dec, xd);
                if (isfinite(r)) q = fma(r, inv_fs, q);
                p = float(q);
            }
            p = __fmul_rn(10.0f, log10f(p));
            pw[i] = p;
            if (p != p || isinf(p)) bad = 1;
            pdb[m] = p;
        }
        const bool ok = !__syncthreads_or(bad);        // any NaN/Inf aborts the update (AFC.h:250-283)
        if (ok) {
            // noise floor = mean, "variance" = standard deviation, both float64 (AFC.h:103-104,225-232); FindPeaks (AFC.h:290-329)
            double s1 = 0;
            float bv = -INFINITY; int bi = 0x7fffffff;
#pragma unroll
            for (int m = 0; m < 16; ++m) {             // ascending shifted index: first maximum wins
                const float p = pdb[m];
                s1 += double(p);
                if (p > bv) { bv = p; bi = t + 256 * m; }
            }
            block_sum_argmax(s1, bv, bi, s_red, 0);
            const double nf = s1 / double(N);
            const float p1v = bv; const int p1 = bi;
            const float rel_sep = float(500.0f / a.fs_dec);
            int sep = int(round(double(rel_sep) * double(N)));
            sep = max(8, sep);
            const int lo = max(p1 - 2 * sep, 0), hi = min(p1 + 2 * sep, N);
            double q = 0;
            bv = -INFINITY; bi = 0x7fffffff;
#pragma unroll
            for (int m = 0; m < 16; ++m) {
                const float p = pdb[m];
                const int i = t + 256 * m;
                const double d = double(p) - nf;
                q += d * d;
                if (i >= lo && i < hi && abs(i - p1) > sep / 2 && p > bv) { bv = p; bi = i; }
            }
            block_sum_argmax(q, bv, bi, s_red, 1);
            if (t == 0) {
                const double nv = sqrt(q / double(N));
                const float P0 = pdb[0];               // thread 0 owns bin 0 of the shifted spectrum
                float p1v_ = p1v, p2v = bv; int p1_ = p1, p2 = bi;
                if (!(p2v > P0)) { p2 = 0; p2v = P0; } // running best starts at v[0], index 0
                if (p2 < p1_) { const int ti = p1_; p1_ = p2; p2 = ti; const float tv = p1v_; p1v_ = p2v; p2v = tv; }
                s_cs.spec_nf = nf; s_cs.spec_nv = nv;
                s_cs.spec_p1 = p1_; s_cs.spec_p2 = p2; s_cs.spec_p1_val = p1v_; s_cs.spec_p2_val = p2v;
            }
        }
        if (t == 0) {
            s_cs.spec_ok = ok ? 1 : 0;
            s_cs.have_spectrum = 1;
            if (s_cs.afc_tick) afc_step(s_cs, a.fs_dec, N);
            st.spec_nf = s_cs.spec_nf; st.spec_nv = s_cs.spec_nv;
            st.spec_p1 = s_cs.spec_p1; st.spec_p2 = s_cs.spec_p2; st.spec_p1_val = s_cs.spec_p1_val; st.spec_p2_val = s_cs.spec_p2_val;
            st.spec_ok = s_cs.spec_ok;
            st.have_spectrum = 1;
            afc_store(st, s_cs);
            st.afc_tick = 0;
            st.fft_ready = 0;
            st.fft_have = 0;
        }
    }
}

// N = 4096 (the reference's fft_bins_cnt_, Decoder.h:163) or 16384 (the 16k-bin spectrum of BASELINE configs[1]:
// four 4096-point sub-transforms of the decimated-by-4 phases + one radix-4 combining pass, all in shared memory).
template <int N>
__global__ void __launch_bounds__(kFftThreads)
fft_afc_kernel(FftArgs a)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* s_a = reinterpret_cast<float2*>(smem_raw);          // exchange area of the 4096-point transform
    float2* s_f = s_a + 16 * 16 * 17;                           // N == 16384: the four sub-spectra [4][4096]
    float* s_p = reinterpret_cast<float*>(s_a + 16 * 16 * 17);  // N == 4096: power spectrum (4096 floats)
    __shared__ double s_red[kFftThreads / 32];
    __shared__ float s_av[kFftThreads / 32];
    __shared__ int s_ai[kFftThreads / 32];
    __shared__ int s_bad;

    __shared__ unsigned char s_todo[kFftThreads];
    const int t = threadIdx.x;
    // CTA b owns channels b, b + G, b + 2G, ... (G = gridDim.x, at most kFftThreads of them).  Phase A: thread j looks at
    // the j-th owned channel; a channel without a complete frame only needs the per-call AFC step (the common case:
    // 15 of 16 calls at 256 decimated samples per call), done here by one thread per channel, all channels in parallel.
    // Phase B: channels with a complete frame are transformed one after the other by the whole CTA.  A small grid with
    // in-CTA ownership keeps the number of 50 KB-shared-memory CTAs that must find room next to the resident K1 small.
    {
        const int j_ch = int(blockIdx.x) + t * int(gridDim.x);
        unsigned char todo = 0;
        if (j_ch < a.n_channels) {
            ChanState& sj = a.state[a.ch0 + j_ch];
            if (sj.fft_ready) todo = 1;
            else if (sj.afc_tick) { afc_step(sj, a.fs_dec, N); sj.afc_tick = 0; }
        }
        s_todo[t] = todo;
    }
    __syncthreads();
    for (int j = 0; int(blockIdx.x) + j * int(gridDim.x) < a.n_channels; ++j) {
    if (!s_todo[j]) continue;
    const int ch = a.ch0 + int(blockIdx.x) + j * int(gridDim.x);
    ChanState& st = a.state[ch];
    const bool do_tick = st.afc_tick != 0;
    __syncthreads();   // everybody has read the flags thread 0 clears at the end of the previous channel

    {
        const float2* x = a.fftbuf + (size_t)ch * N;
        const float2* __restrict__ tw = a.twiddle; // tw[e] = exp(-2 pi i e / N)
        float2* spec = a.spectrum + (size_t)ch * N;
        float* pw = a.power + (size_t)ch * N;
        if (t == 0) s_bad = 0;
        int bad = 0;
        const double inv_fs = 1.0 / a.fs_dec;
        // FftPower of one bin (AFC.h:236-286), spectrum out with the halves swapped (FFT.cpp:77-87)
        auto emit = [&](int k, float2 z) {
            const int i = (k + N / 2) & (N - 1);
            spec[i] = z;
            if (z.x != z.x || z.y != z.y || isinf(z.x) || isinf(z.y)) bad = 1;
            float p = __fadd_rn(__fmul_rn(z.x, z.x), __fmul_rn(z.y, z.y)) / float(N);
            p = __fmul_rn(p, p);
            {   // float(double(p) / fs_dec) (AFC.h:268): reciprocal + one residual step instead of the ~40-instruction
                // IEEE division routine (this line alone was 12 % of the kernel's instructions); the quotient is the
                // correctly rounded one except for double-precision ties that cannot survive the rounding to float
                const double x = double(p);
                double q = x * inv_fs;
                const double r = fma(-q, a.fs_dec, x);
                if (isfinite(r)) q = fma(r, inv_fs, q);
                p = float(q);
            }
            p = __fmul_rn(10.0f, log10f(p));
            if (N == 4096) s_p[i] = p; else pw[i] = p;
        };
        if (N == 4096) {
            fft4096(x, 1, 0, tw + N, tw + N + 4096, s_a, [&](int, int k, float2 z) { emit(k, z); });
        } else {
            for (int r = 0; r < 4; ++r) {
                fft4096(x, 4, r, tw + N, tw + N + 4096, s_a, [&](int, int k, float2 z) { s_f[r * 4096 + k] = z; });
                __syncthreads();
            }
            // X[k + 4096 q] = sum_r W_N^(r k) F_r[k] W_4^(r q)
            for (int k = t; k < 4096; k += kFftThreads) {
                float2 y0 = s_f[k], y1 = cmul(s_f[4096 + k], tw[k]), y2 = cmul(s_f[8192 + k], tw[2 * k]), y3 = cmul(s_f[12288 + k], tw[3 * k]);
                dft4(y0, y1, y2, y3);
                emit(k, y0); emit(k + 4096, y1); emit(k + 8192, y2); emit(k + 12288, y3);
            }
        }
        if (bad) s_bad = 1;
        __syncthreads();
        const float* P = (N == 4096) ? s_p : pw;   // N == 16384: the dB values are re-read from HBM/L2 (written by this CTA)
        int bad2 = 0;
        if (!s_bad) {
            for (int i = t; i < N; i += kFftThreads) {
                const float p = P[i];
                if (N == 4096) pw[i] = p;
                if (p != p || isinf(p)) bad2 = 1;
            }
        }
        if (bad2) s_bad = 1;
        __syncthreads();
        const bool ok = !s_bad;
        if (ok) {
            // noise floor = mean, "variance" = standard deviation, both float64 (AFC.h:103-104,225-232)
            double s = 0;
            for (int i = t; i < N; i += kFftThreads) s += double(P[i]);
            const double nf = block_sum(s, s_red) / double(N);
            double q = 0;
            for (int i = t; i < N; i += kFftThreads) { const double d = double(P[i]) - nf; q += d * d; }
            const double nv = sqrt(block_sum(q, s_red) / double(N));
            // FindPeaks (AFC.h:290-329)
            float bv = -INFINITY; int bi = 0x7fffffff;
            for (int i = t; i < N; i += kFftThreads) { const float p = P[i]; if (p > bv) { bv = p; bi = i; } }
            float p1v; int p1;
            block_argmax(bv, bi, s_av, s_ai, p1v, p1);
            const float rel_sep = float(500.0f / a.fs_dec);
            int sep = int(round(double(rel_sep) * double(N)));
            sep = max(8, sep);
            const int lo = max(p1 - 2 * sep, 0), hi = min(p1 + 2 * sep, N);
            bv = -INFINITY; bi = 0x7fffffff;
            for (int i = lo + t; i < hi; i += kFftThreads) {
                const float p = P[i];
                if (abs(i - p1) > sep / 2 && p > bv) { bv = p; bi = i; }
            }
            float p2v; int p2;
            block_argmax(bv, bi, s_av, s_ai, p2v, p2);
            if (t == 0) {
                if (!(p2v > P[0])) { p2 = 0; p2v = P[0]; } // running best starts at v[0], index 0
                if (p2 < p1) { const int ti = p1; p1 = p2; p2 = ti; const float tv = p1v; p1v = p2v; p2v = tv; }
                st.spec_nf = nf; st.spec_nv = nv;
                st.spec_p1 = p1; st.spec_p2 = p2; st.spec_p1_val = p1v; st.spec_p2_val = p2v;
            }
        }
        if (t == 0) {
            st.spec_ok = ok ? 1 : 0;
            st.have_spectrum = 1;
            st.fft_ready = 0;
            st.fft_have = 0;
        }
        __syncthreads();
    }
    if (do_tick && t == 0) {
        afc_step(st, a.fs_dec, N);
        st.afc_tick = 0;
    }
    }
}

template <int N>
static cudaError_t launch_fft_n(const FftArgs& a, int n_channels, cudaStream_t stream, int* launches)
{
    const size_t smem = size_t(16 * 16 * 17) * 8 + (N == 4096 ? size_t(0) : size_t(16384) * 8);
    static bool configured = false;
    if (!configured) {
        cudaError_t e = N == 4096 ? cudaFuncSetAttribute(fft_afc4096_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                                  : cudaFuncSetAttribute(fft_afc_kernel<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        if (N == 4096) cudaFuncSetAttribute(fft_afc4096_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        else cudaFuncSetAttribute(fft_afc_kernel<N>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        configured = true;
    }
    static int n_sms = 0;
    if (!n_sms) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&n_sms, cudaDevAttrMultiProcessorCount, dev); if (n_sms < 1) n_sms = 1; }
    int grid = std::min(n_channels, 3 * n_sms);   // 3 CTAs per SM are resident (80 registers x 256 threads): one wave
    grid = std::max(grid, (n_channels + kFftThreads - 1) / kFftThreads);   // a CTA owns at most kFftThreads channels
    if (grid < 1) return cudaSuccess;
    FftArgs b = a; b.n_channels = n_channels;
    if (N == 4096) fft_afc4096_kernel<<<grid, kFftThreads, smem, stream>>>(b);
    else fft_afc_kernel<N><<<grid, kFftThreads, smem, stream>>>(b);
    if (launches) ++*launches;
    return cudaGetLastError();
}

cudaError_t launch_fft_afc(const FftArgs& a, int n_channels, cudaStream_t stream, int* launches)
{
    if (a.fft_n == 16384) return launch_fft_n<16384>(a, n_channels, stream, launches);
    return launch_fft_n<4096>(a, n_channels, stream, launches);   // fft_afc4096_kernel
}

// hbd_reset_frequency_correction, one thread per call
__global__ void afc_reset_kernel(ChanState* state, int ch, double corr, double fs_dec, int n_fft)
{
    afc_reset(state[ch], corr, fs_dec, n_fft);
}

cudaError_t launch_afc_reset(ChanState* state, int ch, double corr, double fs_dec, int n_fft, cudaStream_t stream)
{
    afc_reset_kernel<<<1, 1, 0, stream>>>(state, ch, corr, fs_dec, n_fft);
    return cudaGetLastError();
}

// The retune decision of DECODER_THREAD (code/websocketServer/main.cpp:248-265) for every channel at once: where
// |frequency_correction| exceeds min_abs_hz the correction is handed to the caller (who adds it to the channel's
// NCO) and the AFC is reset exactly like resetFrequencyCorrection(); applied[ch] = 0 elsewhere.
__global__ void afc_retune_kernel(ChanState* state, int n_ch, double min_abs_hz, double fs_dec, double* applied, int n_fft)
{
    const int ch = blockIdx.x * blockDim.x + threadIdx.x;
    if (ch >= n_ch) return;
    ChanState& st = state[ch];
    const double corr = st.afc_correction;
    if (!(min_abs_hz < fabs(corr))) { applied[ch] = 0.0; return; }
    applied[ch] = corr;
    afc_reset(st, corr, fs_dec, n_fft);
}

cudaError_t launch_afc_retune(ChanState* state, int n_ch, double min_abs_hz, double fs_dec, double* applied, int n_fft, cudaStream_t stream)
{
    afc_retune_kernel<<<(n_ch + 127) / 128, 128, 0, stream>>>(state, n_ch, min_abs_hz, fs_dec, applied, n_fft);
    return cudaGetLastError();
}

} // namespace hbd
