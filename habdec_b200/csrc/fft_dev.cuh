// Register-resident FFT building blocks shared by K4 (fft_afc.cu) and the wideband scanner (scan.cu).
//
// 4096 = 16 x 16 x 16: three radix-16 passes (each a 4x4 radix-4 butterfly), 256 threads x 16 points, two exchanges
// through shared memory (the second one padded so both the write and the transposed read are conflict free).  Twiddles
// come from tables evaluated in float64 on the host.  No cuFFT.
#pragma once
#include "hbd_common.cuh"

namespace hbd {

constexpr int kFftThreads = 256;

__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ float2 cmul(float2 a, float2 b) { return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }

// forward 4-point DFT, natural order out
__device__ __forceinline__ void dft4(float2& a0, float2& a1, float2& a2, float2& a3)
{
    const float2 t0 = cadd(a0, a2), t1 = csub(a0, a2), t2 = cadd(a1, a3), t3 = csub(a1, a3);
    a0 = cadd(t0, t2);
    a2 = csub(t0, t2);
    a1 = make_float2(t1.x + t3.y, t1.y - t3.x);
    a3 = make_float2(t1.x - t3.y, t1.y + t3.x);
}

// forward 16-point DFT in registers; output X[c + 4d] is left in v[4c + d]
__device__ __forceinline__ void dft16(float2 (&v)[16])
{
#pragma unroll
    for (int b = 0; b < 4; ++b) dft4(v[b], v[4 + b], v[8 + b], v[12 + b]);
    // W16^e = exp(-2 pi i e / 16)
    const float c1 = 0.92387953251128673848f, s1 = 0.38268343236508978178f, r2 = 0.70710678118654752440f;
    const float2 w1 = make_float2(c1, -s1), w2 = make_float2(r2, -r2), w3 = make_float2(s1, -c1);
    const float2 w6 = make_float2(-r2, -r2), w9 = make_float2(-c1, s1);
    v[5] = cmul(v[5], w1);   // c=1,b=1
    v[6] = cmul(v[6], w2);   // c=1,b=2
    v[7] = cmul(v[7], w3);   // c=1,b=3
    v[9] = cmul(v[9], w2);   // c=2,b=1
    v[10] = make_float2(v[10].y, -v[10].x); // c=2,b=2: W16^4 = -i
    v[11] = cmul(v[11], w6); // c=2,b=3
    v[13] = cmul(v[13], w3); // c=3,b=1
    v[14] = cmul(v[14], w6); // c=3,b=2
    v[15] = cmul(v[15], w9); // c=3,b=3
#pragma unroll
    for (int c = 0; c < 4; ++c) dft4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
}
// index of DFT bin k (0..15) inside v[] after dft16
__device__ __forceinline__ constexpr int bin16(int k) { return 4 * (k & 3) + (k >> 2); }

// 4096-point forward DFT of load(n) (n = 0 .. 4095) by 256 threads: three register-resident radix-16 passes, two exchanges
// through s_a (16*16*17 float2).  tw1 / tw2: the twiddles of pass 1 / 2 in the order the threads read them (host tables
// behind the N-point table, see alloc_fft).  Bin k is handed to store(j2, k, value) with k = k1 + 16*j1 + 256*j2 and j2 a
// compile-time constant after unrolling.
template <typename Load, typename Store>
__device__ __forceinline__ void fft4096_load(Load load, const float2* __restrict__ tw1, const float2* __restrict__ tw2, float2* s_a, Store store)
{
    const int t = threadIdx.x;
    float2 v[16];
    // pass 1: n = 256*n1 + t, DFT over n1 -> k1; twiddle W_4096^(t*k1); A[k1][t]
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = load(256 * i + t);
    dft16(v);
#pragma unroll
    for (int k1 = 0; k1 < 16; ++k1) {
        float2 y = v[bin16(k1)];
        if (k1) y = cmul(y, tw1[k1 * 256 + t]);          // W_4096^(t*k1), table laid out [k1][t]: coalesced
        s_a[k1 * 256 + t] = y;
    }
    __syncthreads();
    // pass 2: thread (k1, m2): n2 = 16*m1 + m2, DFT over m1 -> j1; twiddle W_256^(m2*j1); B[k1][j1][m2] (row pitch 17)
    {
        const int k1 = t >> 4, m2 = t & 15;
#pragma unroll
        for (int i = 0; i < 16; ++i) v[i] = s_a[k1 * 256 + 16 * i + m2];
        dft16(v);
        __syncthreads();
#pragma unroll
        for (int j1 = 0; j1 < 16; ++j1) {
            float2 y = v[bin16(j1)];
            if (j1) y = cmul(y, tw2[j1 * 16 + m2]);           // W_256^(m2*j1), [j1][m2]
            s_a[k1 * (16 * 17) + j1 * 17 + m2] = y;
        }
    }
    __syncthreads();
    // pass 3: thread (k1, j1): DFT over m2 -> j2; X[k1 + 16*j1 + 256*j2]
    {
        const int k1 = t >> 4, j1 = t & 15;
#pragma unroll
        for (int i = 0; i < 16; ++i) v[i] = s_a[k1 * (16 * 17) + j1 * 17 + i];
        dft16(v);
        __syncthreads();
#pragma unroll
        for (int j2 = 0; j2 < 16; ++j2) store(j2, k1 + 16 * j1 + 256 * j2, v[bin16(j2)]);
    }
}

// the same transform of x[stride * n + offset]
template <typename Store>
__device__ __forceinline__ void fft4096(const float2* __restrict__ x, int stride, int offset, const float2* __restrict__ tw1,
                                        const float2* __restrict__ tw2, float2* s_a, Store store)
{
    fft4096_load([&](int n) { return x[(size_t)stride * n + offset]; }, tw1, tw2, s_a, store);
}

} // namespace hbd
