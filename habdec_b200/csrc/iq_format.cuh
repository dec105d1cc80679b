// Input sample formats (include/habdec_b200.h, HBD_IQ_*) and their dequantisation on the device.
//
//   CF32  8 B  float I, Q               as is
//   CS16  4 B  int16 I, Q  (LE)         v / 32768
//   CS8   2 B  int8 I, Q                v / 128
//   CU8   2 B  uint8 I, Q  (rtl_sdr)    (v - 128) / 128   (CS8 of v ^ 0x80)
//
// Every value is exactly representable in float32, so an integer push is bit for bit the cf32 push of its dequantised
// values.  The conversion is an exact bit construction instead of I2F (a quarter-rate conversion unit): the biased code
// u (0 .. 2^k - 1) is placed in the low mantissa bits of 2^e whose ulp is the format's scale (PRMT, ALU pipe), and one
// packed FADD2 removes the bias 2^e + 1:  (2^e + u 2^-s) - (2^e + 1) = (u - 2^s) 2^-s, exact (Sterbenz).
#pragma once
#include "hbd_common.cuh"
#include "../../include/habdec_b200.h"

namespace hbd {

inline int iq_bytes(int format)   // bytes per complex sample, 0: unknown format
{
    switch (format) {
    case HBD_IQ_CF32: return 8;
    case HBD_IQ_CS16: return 4;
    case HBD_IQ_CS8:
    case HBD_IQ_CU8: return 2;
    default: return 0;
    }
}

template <int F> struct IqFmt;
template <> struct IqFmt<HBD_IQ_CF32> {
    using T = float2;
#ifdef __CUDACC__
    static __device__ __forceinline__ float2 dq(float2 x) { return x; }
#endif
};
template <> struct IqFmt<HBD_IQ_CS16> {
    using T = uint32_t;   // I in the low half, Q in the high half
#ifdef __CUDACC__
    static __device__ __forceinline__ float2 dq(uint32_t w)
    {
        const uint32_t u = w ^ 0x80008000u;   // biased codes v + 32768
        return cadd2(make_float2(__uint_as_float(__byte_perm(u, 0x43800000u, 0x7610)), __uint_as_float(__byte_perm(u, 0x43800000u, 0x7632))),
                     make_float2(-257.f, -257.f));   // 2^8 + u 2^-15 - (2^8 + 1)
    }
#endif
};
template <int Flip> struct IqByte {
    using T = uint16_t;   // I in the low byte, Q in the high byte
#ifdef __CUDACC__
    static __device__ __forceinline__ float2 dq(uint16_t h)
    {
        const uint32_t u = uint32_t(h) ^ uint32_t(Flip);   // biased codes v + 128
        return cadd2(make_float2(__uint_as_float(__byte_perm(u, 0x47800000u, 0x7640)), __uint_as_float(__byte_perm(u, 0x47800000u, 0x7641))),
                     make_float2(-65537.f, -65537.f));   // 2^16 + u 2^-7 - (2^16 + 1)
    }
#endif
};
template <> struct IqFmt<HBD_IQ_CS8> : IqByte<0x8080> {};
template <> struct IqFmt<HBD_IQ_CU8> : IqByte<0> {};

} // namespace hbd
