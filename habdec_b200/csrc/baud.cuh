// Keying-rate estimator (baud.cu): per channel, a histogram of the debounced sign-run lengths of the discriminator output,
// scored against the usual RTTY rates when the caller asks.  The estimator is stated in include/habdec_b200.h.
#pragma once
#include <algorithm>
#include <cmath>

#include "../../include/habdec_b200.h"
#include "hbd_common.cuh"

namespace hbd {

// A channel's edge state.  Positions count discriminator samples since the estimator (re)started; all zero is a
// restarted estimator.
struct BaudTrack {
    unsigned long long pos;            // samples seen
    unsigned long long streak_start;   // first sample of the current opposite-sign streak
    unsigned long long last_edge;      // position of the last accepted edge
    unsigned streak;                   // length of that streak (0: none)
    unsigned flags;                    // kBaudStarted | kBaudPositive | kBaudHaveEdge
    unsigned long_runs;                // runs longer than the histogram
    unsigned pad_;
};
enum : unsigned { kBaudStarted = 1u, kBaudPositive = 2u, kBaudHaveEdge = 4u };

// What the estimator derives from fs_dec: histogram length Lmax = ceil(6.5 fs / 50), debounce m = max(1, floor(fs / 2400))
struct BaudGeometry { int lmax, m; };
inline BaudGeometry baud_geometry(double fs)
{
    return {int(std::ceil(6.5 * fs / 50)), std::max(1, int(std::floor(fs / 2400)))};
}

struct BaudHistArgs {
    const ChanPlan* plan;   // per-channel plans (read only when !uniform)
    ChanPlan uplan;
    int uniform;
    const ChanState* state; // n_filtered: the discriminator samples the tail kernel produced in this call
    const float* demod; size_t demod_pitch;
    unsigned* hist; size_t hist_pitch;   // [channel][Lmax + 1]
    BaudTrack* track;
    int lmax, m;
};

// once per call with estimation on, behind the tail kernel on its stream
cudaError_t launch_baud_hist(const BaudHistArgs& a, int n_channels, cudaStream_t stream, int* launches);
// on query: one hbd_baud_estimate per channel into out[n_channels]
cudaError_t launch_baud_score(const unsigned* hist, size_t hist_pitch, int lmax, const BaudTrack* track, double fs,
                              hbd_baud_estimate* out, int n_channels, cudaStream_t stream);

} // namespace hbd
