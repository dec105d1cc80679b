// Keying-rate estimator (include/habdec_b200.h, "baud-rate estimation"): the run histograms, stepped once per call behind
// the tail kernel, and the scoring of them against the candidate rates, run on query.
#include "baud.cuh"

namespace hbd {

namespace {

constexpr int kHistWarps = 4;      // channels per CTA of baud_hist_kernel (one warp each)
constexpr int kScoreThreads = 256;
constexpr int kCands = 7;
__constant__ double kCandBaud[kCands] = {50, 75, 100, 150, 200, 300, 600};

// One warp per channel.  The lanes load 32 consecutive samples and ballot their signs; the warp then walks the debounced
// edges of that word with find-first-set, every lane the same way (the walk is warp-uniform), and lane 0 counts the runs.
__global__ void __launch_bounds__(kHistWarps * 32) baud_hist_kernel(BaudHistArgs a, int n_ch)
{
    const int lane = threadIdx.x & 31, ch = blockIdx.x * kHistWarps + (threadIdx.x >> 5);
    if (ch >= n_ch) return;
    const unsigned flags_plan = a.uniform ? a.uplan.flags : a.plan[ch].flags;
    if (flags_plan & 1u) return;   // the tail kernel returned early: n_filtered is an earlier call's
    const unsigned nf = a.state[ch].n_filtered;
    if (!nf) return;
    const float* d = a.demod + size_t(ch) * a.demod_pitch;
    unsigned* H = a.hist + size_t(ch) * a.hist_pitch;
    BaudTrack t = a.track[ch];
    const unsigned m = unsigned(a.m);
    const unsigned long long lmax = (unsigned long long)a.lmax;
    for (unsigned base = 0; base < nf; base += 32) {
        const unsigned n = min(32u, nf - base);
        const unsigned w = __ballot_sync(~0u, base + lane < nf && d[base + lane] > 0.f);   // a zero counts as negative
        const unsigned valid = n == 32 ? ~0u : (1u << n) - 1u;
        if (!(t.flags & kBaudStarted)) t.flags = kBaudStarted | ((w & 1u) ? kBaudPositive : 0u);
        unsigned x = ((t.flags & kBaudPositive) ? ~w : w) & valid;   // samples of the opposite sign
        unsigned j = 0;
        while (j < n) {
            if (!t.streak) {   // the next opposite-sign sample starts a streak
                const unsigned y = x >> j;
                if (!y) break;
                j += unsigned(__ffs(int(y))) - 1u;
                t.streak_start = t.pos + j;
            }
            const unsigned z = ~(x >> j);
            const unsigned run = z ? unsigned(__ffs(int(z))) - 1u : 32u;   // opposite-sign samples from j on (x is 0 beyond n)
            if (t.streak + run >= m) {   // edge at the streak's first sample
                if (t.flags & kBaudHaveEdge) {
                    const unsigned long long L = t.streak_start - t.last_edge;
                    // a fire-and-forget add: the row has this one writer, and the walk need not wait for the load
                    if (L >= 1 && L <= lmax) { if (lane == 0) atomicAdd(H + L, 1u); }
                    else ++t.long_runs;
                }
                t.last_edge = t.streak_start;
                t.flags = (t.flags | kBaudHaveEdge) ^ kBaudPositive;
                x = ~x & valid;
                j += m - t.streak;
                t.streak = 0;
            } else if (j + run >= n) {   // the streak goes on into the next word
                t.streak += run;
                break;
            } else {                     // too short: discarded
                t.streak = 0;
                j += run;
            }
        }
        t.pos += n;
    }
    if (lane == 0) a.track[ch] = t;
}

// One CTA per channel: E(b), sum(H k) and sum(H L) of every candidate over the bins, reduced in uint64; thread 0 picks.
// The tolerance test is written out in round-to-nearest operations so that it is not contracted into FMAs.
__global__ void __launch_bounds__(kScoreThreads) baud_score_kernel(const unsigned* __restrict__ hist, size_t pitch, int lmax,
                                                                   const BaudTrack* __restrict__ track, double fs,
                                                                   hbd_baud_estimate* __restrict__ out)
{
    constexpr int kVals = 3 * kCands + 1;   // E, sum H k, sum H L per candidate, then runs
    __shared__ unsigned long long red[kScoreThreads / 32][kVals];
    const int ch = blockIdx.x, tid = threadIdx.x;
    const unsigned* H = hist + size_t(ch) * pitch;
    int nc = 0;
    while (nc < kCands && fs / kCandBaud[nc] >= 8.0) ++nc;   // the candidates ascend: fs / b >= 8 holds for a prefix
    unsigned long long v[kVals];
#pragma unroll
    for (int i = 0; i < kVals; ++i) v[i] = 0;
    for (int L = 1 + tid; L <= lmax; L += kScoreThreads) {
        const unsigned h = H[L];
        if (!h) continue;
        v[kVals - 1] += h;
        const double Ld = double(L);
#pragma unroll
        for (int c = 0; c < kCands; ++c) {
            if (c >= nc) break;
            const double sp = fs / kCandBaud[c];
            const double k = floor(__dadd_rn(__ddiv_rn(Ld, sp), 0.5));
            if (k < 1.0 || k > 6.0) continue;
            if (fabs(__dsub_rn(Ld, __dmul_rn(k, sp))) > __dmul_rn(0.2, sp)) continue;
            v[3 * c] += h;
            v[3 * c + 1] += (unsigned long long)h * (unsigned long long)k;
            v[3 * c + 2] += (unsigned long long)h * (unsigned long long)L;
        }
    }
#pragma unroll
    for (int i = 0; i < kVals; ++i) {
        for (int o = 16; o; o >>= 1) v[i] += __shfl_down_sync(~0u, v[i], o);
        if ((tid & 31) == 0) red[tid >> 5][i] = v[i];
    }
    __syncthreads();
    if (tid) return;
#pragma unroll
    for (int i = 0; i < kVals; ++i) {
        v[i] = 0;
        for (int w = 0; w < kScoreThreads / 32; ++w) v[i] += red[w][i];
    }
    hbd_baud_estimate e{};
    const unsigned long long runs = v[kVals - 1];
    e.runs = unsigned(runs);
    e.long_runs = track[ch].long_runs;
    if (runs && nc) {
        unsigned long long emax = 0;
#pragma unroll
        for (int c = 0; c < kCands; ++c) if (c < nc) emax = max(emax, v[3 * c]);
        // the lowest rate within 90 % of the best, not a harmonic of it (descending: the last match is the lowest)
        int pick = 0;
        unsigned long long E = 0, SK = 0, SL = 0;
#pragma unroll
        for (int c = kCands - 1; c >= 0; --c)
            if (c < nc && 10ull * v[3 * c] >= 9ull * emax) { pick = c; E = v[3 * c]; SK = v[3 * c + 1]; SL = v[3 * c + 2]; }
        e.nominal = kCandBaud[pick];
        e.confidence = __ddiv_rn(double(E), double(runs));
        e.baud = SL ? __ddiv_rn(__dmul_rn(fs, double(SK)), double(SL)) : 0.0;
    }
    out[ch] = e;
}

} // namespace

cudaError_t launch_baud_hist(const BaudHistArgs& a, int n_channels, cudaStream_t stream, int* launches)
{
    baud_hist_kernel<<<(n_channels + kHistWarps - 1) / kHistWarps, kHistWarps * 32, 0, stream>>>(a, n_channels);
    if (launches) ++*launches;
    return cudaGetLastError();
}

cudaError_t launch_baud_score(const unsigned* hist, size_t hist_pitch, int lmax, const BaudTrack* track, double fs,
                              hbd_baud_estimate* out, int n_channels, cudaStream_t stream)
{
    baud_score_kernel<<<n_channels, kScoreThreads, 0, stream>>>(hist, hist_pitch, lmax, track, fs, out);
    return cudaGetLastError();
}

} // namespace hbd
