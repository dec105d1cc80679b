// K1 launch interface (see decim1.cu)
#pragma once
#include "hbd_common.cuh"
#include "nco.cuh"

namespace hbd {

#ifndef HBD_K1_WARPS
#define HBD_K1_WARPS 10
#endif
constexpr int kDecimWarps = HBD_K1_WARPS; // warps per CTA; each warp runs its own TMA ring

struct DecimArgs {
    const float2* chunk;       // pushed samples, [channel][chunk_pitch] cf32 (or the integer format given to launch_decim1), chunk[j] for j in [0, n)
    size_t chunk_pitch;        // in samples, 16-byte rows
    const float2* carry;       // [channel][carry_cap], right aligned: sample j (< 0) at carry[carry_cap + j]
    int carry_cap;             // row length of the carry buffers (>= T1 - 1 + total factor: history + unconsumed remainder)
    float2* s1;                // stage-1 output stream, [channel][s1_pitch]; outputs start at s1_hist
    size_t s1_pitch;
    int s1_hist;
    const ChanPlan* plan;      // per channel (read only when !uniform)
    ChanPlan uplan;            // the plan of every channel when uniform (kernel argument: no upload, no dependent global load)
    int uniform;
    const float* taps;         // T floats (device)
    int ch0;                   // first channel of this launch
    int n_channels;            // channels in this launch
    float2* carry_next;        // other half of the carry ping-pong pair: K1 writes the next call's carry here
    int sb_per_channel;        // superblock slots per channel (uniform upper bound; set by launch_decim1)
    int span;                  // superblocks per warp (contiguous in the flattened (channel, superblock) plane)
    const NcoChan* nco;        // non-null: `chunk` holds RAW samples (chunk_pitch 0: one wideband row shared by all channels) and K1
                               // mixes every channel through its NCO on the fly (fused K0); the carry always holds mixed samples
};

// M == 1 means "no decimator" (copy).  `launches` is incremented per kernel launched.  Writes the carry of the
// next call into a.carry_next (inside K1 on the fast path, by carry_kernel otherwise).  `format` (HBD_IQ_*) is that of
// a.chunk; an integer format needs decim1_supports_native_iq and no NCO.  The carry is cf32 whatever the format.
cudaError_t launch_decim1(DecimArgs a, int M, int T, unsigned max_n1, int n_sms, cudaStream_t stream, int* launches, int format = 0);
// can launch_decim1 mix the channels through their NCOs itself (DecimArgs::nco) for this first stage?
bool decim1_supports_fused_nco(int M, int T);
// can launch_decim1 read integer input (CS16 / CS8 / CU8) itself for this first stage?
bool decim1_supports_native_iq(int M, int T);
// stage-1 carry (history + unconsumed remainder) for the next call: carry -> carry_next
cudaError_t launch_carry(const ChanPlan* plan, ChanPlan uplan, int uniform, const float2* chunk, size_t chunk_pitch, const float2* carry, float2* carry_next, int T1, int ch0,
                         int n_channels, int carry_cap, cudaStream_t stream, int* launches);

} // namespace hbd
