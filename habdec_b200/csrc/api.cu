// C ABI of libhabdec_b200.so (include/habdec_b200.h): handle, HBM state, per-call planning
// (the host mirror of the reference's buffer bookkeeping, Decoder.h:426-436,492-542), kernel
// sequencing and the host sentence layer.  There is no CPU compute path in here: every
// process call launches K1..K4 or fails.
#include "../../include/habdec_b200.h"

#include <algorithm>
#include <array>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <sched.h>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "baud.cuh"
#include "decim1.cuh"
#include "iq_format.cuh"
#include "mid.cuh"
#include "decim_taps.inc"
#include "fft_afc.cuh"
#include "hbd_common.cuh"
#include "host_tail.h"
#include "range_pool.h"
#include "telemetry_abi.h"
#include "api_internal.h"
#include "cuda_res.h"
#include "nco.cuh"
#include "ssdv.cuh"
#include "tail.cuh"
#include "wire.cuh"

using namespace hbd;

namespace {

struct TapTable { int M; const uint32_t* bits; int len; };
#define HBD_TT(M, name) TapTable{M, hbd_taps_bits_##name, int(sizeof(hbd_taps_bits_##name) / 4)}

// factor -> stage list, Decoder.h:286-320
bool plan_for_factor(size_t factor, std::vector<TapTable>& st)
{
    st.clear();
    switch (factor) {
    case 256: st = {HBD_TT(64, d256_m64), HBD_TT(4, d4_m4)}; return true;
    case 128: st = {HBD_TT(32, d128_m32), HBD_TT(4, d4_m4)}; return true;
    case 64:  st = {HBD_TT(32, d64_m32), HBD_TT(2, d2_m2)}; return true;
    case 32:  st = {HBD_TT(16, d32_m16), HBD_TT(2, d2_m2)}; return true;
    case 16:  st = {HBD_TT(8, d16_m8), HBD_TT(2, d2_m2)}; return true;
    case 8:   st = {HBD_TT(8, d8_m8)}; return true;
    case 4:   st = {HBD_TT(4, d4_m4)}; return true;
    case 2:   st = {HBD_TT(2, d2_m2)}; return true;
    case 1:   return true;
    default:  return false;
    }
}

constexpr int kMaxMidStages = 6;   // a cascaded plan has at most 8 stages: K1's, up to six in the middle, the tail kernel's

// host mirror of one channel, part 1: stream counters that are pure functions of the push sizes (and of the
// low-pass configuration).  While every channel is fed the same way they are identical for all channels, and only
// hc[0]'s copy is kept current (hbd_decoder::ctr_uniform / sync_ctrs): a steady-state call costs O(1) host work.
// The FFT frame fill is not among them (HostChan::fft_have, hbd_decoder::fft_lvl): a channel reset in mid-stream
// starts its frame empty while the others are partway through theirs, and agrees with them in everything else.
struct ChanCtr {
    unsigned in_r = 0, dec_pending = 0;
    size_t grown1 = 0, grown2 = 0, grown_lp = 0;
    size_t grown_mid[kMaxMidStages] = {0, 0, 0, 0, 0, 0};   // work-buffer sizes of the middle stages of a cascaded plan
    size_t lp_input_size = 0, lp_ntaps = 0;
    unsigned pushed = 0;     // samples waiting in the staging row
    unsigned last_nf = 0, last_n2 = 0;
    unsigned demod_n = 0;    // size of the reference's demodulated_ (last call that produced any; Decoder.h:546-555)
    bool lp_dirty = true;    // bw / trans / input size changed since the last design attempt
    bool same(const ChanCtr& o) const
    {
        for (int k = 0; k < kMaxMidStages; ++k) if (grown_mid[k] != o.grown_mid[k]) return false;
        return in_r == o.in_r && dec_pending == o.dec_pending && grown1 == o.grown1 && grown2 == o.grown2 && grown_lp == o.grown_lp &&
               lp_input_size == o.lp_input_size && lp_ntaps == o.lp_ntaps && pushed == o.pushed &&
               last_nf == o.last_nf && last_n2 == o.last_n2 && demod_n == o.demod_n && lp_dirty == o.lp_dirty;
    }
};
// part 2: configuration (always per channel)
struct HostChan : ChanCtr {
    double baud = 1;         // SymbolExtractor default symbol_rate_ = 1
    size_t rtty_bits = 0;
    float rtty_stops = 0;
    float lp_bw = 1500, lp_trans = 0.025f;
    bool dc_remove = false;
    double nco_freq = 0, nco_phase = 0; // pre-mixer: frequency in Hz, phase (cycles) of the next pushed sample
    bool cfg_dirty = true;
    // mirror of ChanState::fft_have: tells the host which calls complete an FFT frame (K4 launch).  Current in per-channel
    // mode only; in uniform mode the channel's frame level (hbd_decoder::fft_lvl) holds it.
    unsigned fft_have = 0;
    ChanCtr& ctr() { return *this; }
};

// What one channel's share of a process() call amounts to on the host: the reference's buffer arithmetic
// (Decoder.h:426-436,492-542) stepped on the channel's counters (step_channel), and the side effects that
// hbd_decoder::apply_step applies to that channel's rows -- or, in uniform mode, to the rows of every channel at once.
struct ChanStep {
    ChanPlan plan;
    bool zero_carry = false;       // Decimator.h:74-79: the stage's work buffer grew -> its history is zeroed
    bool zero_s1hist = false;      // ... of the LAST stage (the tail kernel's input buffer)
    unsigned zero_mid = 0;         // bit k: ... of middle stage k (cascaded plans)
    bool zero_lphist = false;      // FirFilter.h:141-147
    bool taps_changed = false;     // low-pass redesigned: upload `taps`
    size_t taps_old = 0, taps_new = 0;
    unsigned nf = 0;
};

// what the kernel launches of a process call read from its planning (plan_call -> enqueue_call)
struct CallPlan {
    ChanPlan uplan{};   // every channel's plan when plan_uniform, else channel 0's (d_plan holds them all)
    bool plan_uniform = true, any_work = false, need_k4 = false;
    unsigned max_n1 = 0;
    int sv_want = 0;
};

constexpr unsigned kMaxCallsBetweenCollects = 256; // process_async forces a drain beyond this (log capacity)

__global__ void init_cfg_kernel(ChanState* st, const double* baud, const float* stops, const int* bits, const int* dc, const int* ntaps,
                                const unsigned char* dirty, int n_ch)
{
    const int ch = blockIdx.x * blockDim.x + threadIdx.x;
    if (ch >= n_ch || !dirty[ch]) return;
    st[ch].baud = baud[ch];
    if (st[ch].rtty_stops != stops[ch] || st[ch].rtty_bits != bits[ch]) st[ch].uart_rescan = 1;   // RTTY.h:90-134 rescans bits_ under the new framing
    st[ch].rtty_stops = stops[ch];
    st[ch].rtty_bits = bits[ch];
    st[ch].dc_remove = dc[ch];
    st[ch].lp_ntaps = ntaps[ch];
}

// ChanState of a newly created decoder: Average<T>'s constructor add()s one 0, so the counts start at 1 (Average.h:34-37);
// the configuration fields are those of a channel no setter has reached yet (the next call's upload fills them in)
__host__ __device__ inline void fresh_state(ChanState& s)
{
    memset(&s, 0, sizeof(s));
    s.baud = 1; // SymbolExtractor.h:96
    s.nf_cnt = s.nv_cnt = s.pl_cnt = s.pr_cnt = 1;
}

// hbd_reset_channels: one CTA per listed channel.  Besides the state it restarts what the next call reads below a count
// it does not find in ChanState: the low-pass work buffer with its stale-input slots (FirFilter.h:139-147 keep them
// for a longer filter), and the per-channel counts of the demod accumulator, the SSDV ring and the recorded bits.
// The carry and stage histories are zeroed by the next call's plan (grown* == 0); every other row is rewritten
// before it is read (FFT frame from fft_have = 0, spectra behind have_spectrum, slicer / mask / UART rows below
// their counts).  With baud estimation on it also restarts the channel's estimator.
struct ResetArgs {
    ChanState* state; const int* list;
    float2* decq; size_t dq_pitch;   // nullptr before the first call sized it
    unsigned* dacc_n; unsigned* ssdv_total; unsigned* ssdv_scanned; unsigned* rec_bits_n;   // the last three may be nullptr
    unsigned* bhist; size_t bhist_pitch; BaudTrack* btrack;   // nullptr while baud estimation has no rows
};
__global__ void reset_chan_kernel(ResetArgs a)
{
    const int ch = a.list[blockIdx.x];
    if (a.decq) for (int i = threadIdx.x; i < kLpHist; i += blockDim.x) a.decq[size_t(ch) * a.dq_pitch + i] = make_float2(0.f, 0.f);
    if (a.bhist) for (size_t i = threadIdx.x; i < a.bhist_pitch; i += blockDim.x) a.bhist[size_t(ch) * a.bhist_pitch + i] = 0u;
    if (threadIdx.x) return;
    if (a.btrack) a.btrack[ch] = BaudTrack{};
    fresh_state(a.state[ch]);
    a.dacc_n[ch] = 0;
    if (a.ssdv_total) { a.ssdv_total[ch] = 0; a.ssdv_scanned[ch] = 0; }
    if (a.rec_bits_n) a.rec_bits_n[ch] = 0;
}

// a channel's AFC scalars in the order of hbd_get_stats_batch and hbd_result_record: correction, shift, noise floor,
// noise variance, peak left, peak right
template <class T>
__host__ __device__ inline void afc_scalars(const ChanState& s, T out[6])
{
    out[0] = T(s.afc_correction); out[1] = T(s.afc_shift_hz); out[2] = T(s.afc_noise_floor); out[3] = T(s.afc_noise_var);
    out[4] = T(s.gui_left); out[5] = T(s.gui_right);
}

// the per-channel scalars that travel with the gathered results (hbd_result_record), packed after every call
__global__ void stats_snap_kernel(const ChanState* __restrict__ st, float* __restrict__ out, int n_ch)
{
    const int ch = blockIdx.x * blockDim.x + threadIdx.x;
    if (ch >= n_ch) return;
    afc_scalars(st[ch], out + size_t(ch) * 6);
}

} // namespace

// a user callback recorded under the handle's mutex and fired after it is released (a callback may call hbd_* again)
struct Deferred {
    enum Kind { kSentence, kChars, kSsdv } kind;
    int ch;
    std::string a, b, c;                                   // sentence: callsign, data, crc; chars: a
    hbd_ssdv_packet_info info; std::array<unsigned char, 256> pkt;
};

// what one thread of the drain records for its channel range (collect_locked)
struct ReplayPart { std::vector<std::pair<unsigned, Deferred>> events; bool spilled = false; };

// the samples of one hbd_push_* call (hbd_decoder::push)
struct PushSrc {
    enum Shape { kChannel, kMatrix, kRow };   // one channel's samples, [n_ch][pitch], one wideband row for all channels
    const void* p;
    bool device;
    int format;     // HBD_IQ_*
    Shape shape;
    int ch;         // kChannel
    size_t pitch;   // kMatrix, in samples
    size_t n;
    double fs;
};

struct hbd_decoder {
    std::mutex mtx;
    std::string err;
    int n_ch = 0, device = 0, n_sms = 148;
    // The streams come first: members are destroyed in reverse order, so the streams outlive the buffers and events.
    cudaStream_t stream = nullptr;   // the caller's stream: inputs are ordered on it, it waits until inputs are consumed
    Stream own_stream;               // the private stream `stream` is until hbd_set_stream
    // Two streams: the HBM-bound K1 of call s+1 overlaps the FP32/latency-bound tail kernels of call s (the stage-1
    // stream and the carry are double buffered over calls, so K1 only ever waits for the tail of call s-1).
    //   hi (high priority): K1 (+ carry) of every call
    //   lo (low priority):  K2 tail / K4 fft_afc; they fill the SM resources K1 leaves free
    Stream hi, lo;
    Stream copy_stream;              // result read-back, independent of the compute streams
    Event ev_consumed;               // K1 + carry done (input consumed, stage-1 output ready)
    Event ev_tail[2];                // per stage-1 buffer: tail done, that buffer may be overwritten by K1
    bool tail_pending[2] = {false, false};
    bool tail_ev_late = false;              // HBD_TAIL_EV_LATE=1 (measurement hook): record ev_tail after the whole lo-stream sequence
    Event ev_in;
    int sync_groups()
    {
        if (hi && cudaStreamSynchronize(hi.get()) != cudaSuccess) return HBD_ERR_CUDA;
        if (lo && cudaStreamSynchronize(lo.get()) != cudaSuccess) return HBD_ERR_CUDA;
        return HBD_OK;
    }
    // wait until everything the handle has enqueued is done: the compute streams, then the caller's stream
    int settle()
    {
        HBD_CUDA_CHECK(cudaSetDevice(device));
        if (sync_groups()) { set_error("stream sync failed"); return HBD_ERR_CUDA; }
        HBD_CUDA_CHECK(cudaStreamSynchronize(stream));
        return HBD_OK;
    }
    // the device state of channels [c0, c0 + n) once everything enqueued is done
    int read_states(size_t c0, size_t n, ChanState* out)
    {
        if (settle()) return HBD_ERR_CUDA;
        HBD_CUDA_CHECK(cudaMemcpy(out, d_state.get() + c0, n * sizeof(ChanState), cudaMemcpyDeviceToHost));
        return HBD_OK;
    }
    ~hbd_decoder()
    {
        settle();
        dist_ctx.reset();
    }
    // plan_call: wait for the compute streams once, before the first host-side change a kernel in flight could see
    bool groups_idle = false;
    int quiesce() { if (!groups_idle) { if (sync_groups()) return HBD_ERR_CUDA; groups_idle = true; } return HBD_OK; }
    bool record = false;
    unsigned long long launches = 0;

    double fs_in = 0;
    int factor = 1;
    int M1 = 1, T1 = 1, M2 = 1, T2 = 1;   // first stage (K1) and last stage (tail kernel; M2 == 1: the plan has one stage)
    struct MidStage { int M = 1, T = 1; unsigned div_in = 1; DevPtr<float> d_taps; Rows<float2> out; };
    std::vector<MidStage> mids;           // stages[1 .. size-2] of the plan (Decoder.h:286-320, cascaded by setupDecimationStagesBW :350-399)
    Rows<float2, 2> midlast;              // output of the last middle stage = the tail kernel's input, ping-pong over calls like s1x
    // The input buffer of middle stage k (k == mids.size(): of the tail kernel): history slots [0, hist), this call's
    // samples from hist on; `next` receives the history for the next call (== p where the buffer is not ping-ponged).
    struct StageRows { float2* p; float2* next; size_t pitch; int hist; };
    StageRows stage_in(size_t k) const
    {
        if (k == 0) return {s1x.get(s1_cur), s1x.get(s1_cur ^ 1), s1x.pitch, kS1Hist};
        if (k < mids.size()) return {mids[k - 1].out.get(), mids[k - 1].out.get(), mids[k - 1].out.pitch, kMidHist};
        return {midlast.get(s1_cur), midlast.get(s1_cur ^ 1), midlast.pitch, kS1Hist};
    }
    int carry_cap = kCarryCapMin;
    int set_plan(const std::vector<TapTable>& st, size_t total_factor);
    int fft_n = kFftN;       // spectrum size: 4096 like the reference, or 16384 (hbd_set_fft_size)
    struct FftBufs { DevPtr<float2> buf, spectrum, twiddle; DevPtr<float> power; } fft;
    int make_fft(int N, FftBufs& out);
    std::vector<HostChan> hc;        // per-channel configuration + counters (see ChanCtr)
    // Uniform mode: every channel has been fed the same way since creation (whole-batch pushes only), so all ChanCtr are
    // equal and only hc[0]'s is stepped per call; hc[1..] lag behind (ctr_stale) until sync_ctrs() copies them.
    bool ctr_uniform = true, ctr_stale = false;
    bool lp_cfg_uniform = true;      // lp_bw / lp_trans are the same for all channels (setters with ch == -1 only)
    bool cfg_dirty_any = true;       // some channel has cfg_dirty set
    bool derived_dirty = true;       // max_lp_taps_c / max_spb_c need recomputing
    size_t max_lp_taps_c = 1; double max_spb_c = 1;
    void sync_ctrs() { if (ctr_stale) { for (size_t c = 1; c < hc.size(); ++c) hc[c].ctr() = hc[0].ctr(); ctr_stale = false; } }
    // FFT frame levels: in uniform mode the distinct frame fills of the channels (fft_lvl) and each channel's index into it
    // (lvl_of).  A uniform call steps every level once; without resets there is exactly one.
    std::vector<unsigned> fft_lvl{0u}, lvl_of;
    void leave_uniform()
    {
        sync_ctrs();
        if (ctr_uniform) for (size_t c = 0; c < hc.size(); ++c) hc[c].fft_have = fft_lvl[lvl_of[c]];
        ctr_uniform = false;
    }
    // back to uniform mode once every channel's ChanCtr agrees again; the frame fills become levels.  O(n log n), called
    // only where the channels have just been stepped or changed one by one.
    void regroup()
    {
        ctr_uniform = true;
        for (size_t c = 1; c < hc.size() && ctr_uniform; ++c) ctr_uniform = hc[c].same(hc[0]);
        if (!ctr_uniform) return;
        fft_lvl.clear();
        for (const HostChan& x : hc) fft_lvl.push_back(x.fft_have);
        std::sort(fft_lvl.begin(), fft_lvl.end());
        fft_lvl.erase(std::unique(fft_lvl.begin(), fft_lvl.end()), fft_lvl.end());
        for (size_t c = 0; c < hc.size(); ++c) lvl_of[c] = unsigned(std::lower_bound(fft_lvl.begin(), fft_lvl.end(), hc[c].fft_have) - fft_lvl.begin());
    }
    double plan_host_ms = 0; unsigned plan_steps = 0;   // host time of plan_call and frame counters it stepped (which = 6)
    // staged (host-pushed, not yet processed) samples: the same count in every channel?
    bool queue_depth_equal(unsigned& base)
    {
        base = hc[0].pushed;
        if (ctr_uniform) return true;
        for (const auto& x : hc) if (x.pushed != base) return false;
        return true;
    }
    void add_pushed(unsigned n)
    {
        if (ctr_uniform) { hc[0].pushed += n; ctr_stale = true; }
        else for (auto& x : hc) x.pushed += n;
    }
    std::vector<TextChannel> text;   // sentence layer state, touched only when a channel produced characters
    bool spill_free = true;                // no channel holds spilled (beyond-the-slot) pending bytes: hbd_pack_results stays sequential
    std::vector<hbd_result_record> pend;   // per channel: characters / sentence bytes waiting for a poll or the next gather (host_tail.h)

    // device state
    DevPtr<ChanState> d_state;
    DevPtr<ChanPlan> d_plan;
    std::vector<ChanPlan> h_plan, h_plan_uploaded;
    DevPtr<float2> d_carry2[2];  // stage-1 carry, ping-pong: K1 reads [carry_cur], writes [carry_cur ^ 1]
    int carry_cur = 0;
    Rows<float2, 2> s1x;         // stage-1 stream, ping-pong over calls:
    int s1_cur = 0;              // K1 + tail of a call use [s1_cur]; the tail leaves the stage-2 history in [s1_cur ^ 1]
    Rows<float2> decq;
    DevPtr<float> d_lptaps;
    Rows<float> slicer, demod;
    DevPtr<unsigned> d_maskc;                // cached slicer position masks [n][2][kMaskWords] (tail.cu)
    DevPtr<unsigned short> d_uart_runs;      // UART backlog [n][kUartRunsCap] (slicer_dev.cuh)
    // Decoded-character log: ring of log_cap entries appended by the tail kernels (monotonic head in d_log_ctl[0]).
    // After the kernels of a call the control words are copied to that call's slot of h_heads (pinned), in stream order:
    // the host only ever reads a COMMITTED head, never the live one (entries below it are completely written).
    DevPtr<uint2> d_log;
    unsigned log_cap = 0;                // power of two, sized from the channel count
    DevPtr<unsigned> d_log_ctl;          // kCtlWords control words (see LogCtl in hbd_common.cuh)
    HostPtr<unsigned> h_heads;           // pinned, [ev_call.size()][kCtlWords]
    HostPtr<unsigned> h_tail_pin;        // pinned, [2]: char log tail, SSDV log tail (source of the async upload)
    unsigned log_tail = 0;               // host: entries below this index are already processed
    unsigned call_seq = 0;               // calls enqueued so far (24 bits travel in the log entries)
    unsigned calls_collected = 0;        // calls whose characters went through the sentence layer
    unsigned done_seq = 0;               // calls known to have completed (event queries, see log_pressure)
    unsigned done_head = 0;              // committed character-log head of call done_seq - 1
    unsigned per_call_max = 0;           // largest number of characters one completed call appended so far
    unsigned long long chars_lost = 0;   // characters dropped by log overflows (reported by hbd_collect*)
    unsigned ovf_seen[3] = {0, 0, 0};    // last seen kCtlSsdvRingOvf / kCtlSsdvOvf / kCtlCharOvf (monotonic counters)
    std::vector<Event> ev_call;          // ring: completion of call (seq % size)
    std::vector<uint2> h_log;           // host staging
    std::vector<std::string> call_chars; // per channel: raw chars of the call being replayed
    std::vector<unsigned> seg_start;     // collect_locked: first log entry of every (call, channel) segment
    static constexpr int kCharBufHost = 64;   // == kCharBuf (slicer_dev.cuh): characters per device-side flush
    double drain_host_ms = 0; unsigned drain_calls = 0;   // host time of the replay part of the drains (hbd_get_kernel_timing which = 5)
    hbd::RangePool pool;                 // the drain's worker threads (part t of a drain / a pack runs on the same thread every time)
    int host_threads = 1;                // threads the drain may use (hbd_set_host_threads; default: min(4, half the cores this process may run on))
    bool keep_raw = true;                // hbd_set_raw_chars: retain the raw (unfiltered) characters for hbd_poll_raw_chars
    DevPtr<float> d_taps1, d_taps2;
    // config upload scratch
    DevPtr<double> d_cfg_baud; DevPtr<float> d_cfg_stops; DevPtr<int> d_cfg_bits, d_cfg_dc, d_cfg_ntaps; DevPtr<unsigned char> d_cfg_dirty;
    // recordings
    Rows<float2, 2> rec;         // [0] decimated, [1] filtered
    DevPtr<unsigned char> d_rec_bits; DevPtr<unsigned> d_rec_bits_n; unsigned rec_bits_pitch = 0;

    // input (push)
    Rows<float2> stage;          // host pushes land here
    // A device push that K1 reads in place at the next process call (p == nullptr: K1 reads the staging matrix).
    // format: integers that K1 reads itself (decim1_supports_native_iq).  nco: raw samples that K1 mixes through the
    // channels' NCOs (fused K0); pitch 0 is one wideband row shared by all channels.
    struct DeviceInput { const void* p = nullptr; size_t pitch = 0, n = 0; int format = HBD_IQ_CF32; const NcoChan* nco = nullptr; } in;
    int push(const PushSrc& s);
    // Host integers are uploaded to iq_up.  d_widen() holds cf32: widened device integers, and wideband rows that do not
    // arrive as device cf32.
    // One row of `pitch` bytes each, grown with grow(bytes, 1, 0, stream): what they held is dropped, and the old buffer is
    // released only after `stream` has caught up (a kernel of an earlier push may still read it).
    Rows<unsigned char> iq_up, widen_buf;
    float2* d_widen() const { return reinterpret_cast<float2*>(widen_buf.get()); }
    int widen(const void* src, size_t pitch, int format, int rows, size_t n, size_t* out_pitch);
    // fused-NCO parameter ring: pinned host slots + device slots, so a push never waits for the GPU
    static constexpr unsigned kNcoSlots = 16;
    HostPtr<NcoChan> h_nco_pin; DevPtr<NcoChan> d_nco_ring; Event ev_nco[kNcoSlots]; unsigned nco_seq = 0;
    bool nco_fused = true;   // HBD_NCO_FUSED=0 (measurement / test hook): always pre-mix with K0 into the staging matrix

    // websocket wire formats (wire.cu)
    bool demod_acc_on = false;
    Rows<float> dacc; DevPtr<unsigned> d_dacc_n;
    DevPtr<unsigned char> d_frames; size_t frames_pitch = 0; DevPtr<unsigned> d_frame_sizes;
    std::vector<unsigned> h_frame_sizes;
    int ensure_frames(size_t pitch);
    int ensure_dacc();
    // NCO pre-mixer (nco.cu)
    DevPtr<NcoChan> d_nco; std::vector<NcoChan> h_nco;
    bool nco_any = false;    // some channel has (had) a non-zero NCO frequency or phase (set by hbd_set_nco, never cleared)
    void nco_params(NcoChan* out, int c0, int nc, size_t n, bool k0_rotation);
    int mix_into_stage(const void* src, size_t src_pitch, int c0, int nc, size_t dst_off, size_t n, int format = HBD_IQ_CF32);
    int sv_override = -1;
    bool mask_cache = true;      // HBD_MASK_CACHE=0 (test hook): the slicer's position masks are rebuilt from scratch in every call
    // optional per-kernel CUDA-event timing (bench roofline): one event pair per K1 launch / per rest-of-step
    int timing = 0;          // 0 off, 1: events around K1 only (what the roofline needs), 2: also around the rest of the step (pipeline diagnostics)
    std::vector<Event> ev_k1, ev_rest;   // pairs: [2i] start, [2i+1] stop
    size_t ev_used_k1 = 0, ev_used_rest = 0;
    cudaEvent_t next_event(std::vector<Event>& pool, size_t& used)
    {
        if (used == pool.size()) { pool.emplace_back(); event_create(pool.back(), cudaEventDefault); }
        return pool[used++].get();
    }
    size_t cap_n_in = 0;     // largest (r + n) the per-call buffers are sized for

    // SSDV packet sync (ssdv.cu + host_tail.cpp SsdvChannel); off until hbd_set_ssdv / hbd_set_ssdv_callback
    bool ssdv_on = false;
    DevPtr<unsigned char> d_ssdv_ring; DevPtr<unsigned> d_ssdv_total, d_ssdv_scanned;
    DevPtr<SsdvLogEntry> d_ssdv_log; unsigned ssdv_log_tail = 0;
    std::vector<SsdvLogEntry> h_ssdv_log;
    std::vector<SsdvChannel> ssdv;
    hbd_ssdv_cb ssdv_cb = nullptr; void* ssdv_user = nullptr;
    int enable_ssdv(bool on);

    hbd_sentence_cb sentence_cb = nullptr; void* sentence_user = nullptr;
    hbd_tracker* tracker = nullptr; int tracker_off = 0;   // telemetry layer fed after the sentence callback
    hbd_chars_cb chars_cb = nullptr; void* chars_user = nullptr;
    std::vector<Deferred> deferred;  // callbacks recorded by collect_locked, fired by the entry point after unlocking
    // result gather (gather.cpp / dist.cu): AFC scalars of every channel snapshotted after each call into a small device
    // ring, so that a drain can read the values that belong to the calls it drains without stopping the pipeline
    static constexpr unsigned kSnapSlots = 32;
    bool snap_on = false;
    DevPtr<float> d_snap;            // [kSnapSlots][n][6]
    HostPtr<float> h_snap;           // pinned, [n][6]: snapshot of the newest drained call
    bool h_snap_valid = false;
    DistSlot dist_ctx;               // dist.cu
    int enable_snap();

    // baud-rate estimation (baud.cu); off until hbd_set_baud_estimation, and then without rows until fs_dec is known
    bool baud_on = false;
    double baud_fs = 0;                  // fs_dec the rows were sized and zeroed for; 0: the estimator restarts at its next use
    int baud_lmax = 0;
    DevPtr<unsigned> d_bhist;            // run histograms [n][baud_lmax + 1]
    DevPtr<BaudTrack> d_btrack;          // edge state [n]
    DevPtr<hbd_baud_estimate> d_best;    // the score kernel's output [n]
    int baud_start();
    int baud_estimates(std::vector<hbd_baud_estimate>& out);

    void set_error(const std::string& e) { err = e; }
    int ensure_call_capacity(size_t n_in_max);
    int alloc_fixed();
    int apply_step(const ChanStep& st, size_t c0, size_t rows, const std::vector<float>& taps);
    int plan_call(CallPlan& cp);
    int enqueue_call(const CallPlan& cp);
    int process_async_locked();
    int collect_locked(unsigned lag);
    HostPtr<int> h_reset; DevPtr<int> d_reset;   // channel list of hbd_reset_channels (allocated by the first one)
    int reset_channels(const int* chs, size_t k);
    int log_pressure();
};

// Runs `body` (a lambda returning int) under the handle's mutex, then fires the callbacks it recorded with the mutex
// released -- a callback may call any hbd_* function of the same handle (the reference's getRTTY()/getLastSentence()
// are callable from sentence_callback_ as well).
namespace {
struct CallbackSet { hbd_sentence_cb s; void* su; hbd_chars_cb c; void* cu; hbd_ssdv_cb v; void* vu; hbd_tracker* trk; int off; };
void fire_deferred(const std::vector<Deferred>& ev, const CallbackSet& cb)
{
    for (const Deferred& d : ev) {
        switch (d.kind) {
        case Deferred::kSentence:
            if (cb.s) cb.s(cb.su, d.ch, d.a.c_str(), d.b.c_str(), d.c.c_str());
            if (cb.trk) tracker_feed(cb.trk, d.ch + cb.off, d.a, d.b, d.c);      // SentenceCallback, websocketServer/main.cpp:292-366
            break;
        case Deferred::kChars: if (cb.c) cb.c(cb.cu, d.ch, d.a.data(), d.a.size()); break;
        case Deferred::kSsdv: if (cb.v) cb.v(cb.vu, d.ch, &d.info, d.pkt.data()); break;
        }
    }
}
template <typename F>
int locked_then_fire(hbd_decoder* h, F body)
{
    std::vector<Deferred> ev;
    CallbackSet cb{};
    int rc;
    {
        std::lock_guard<std::mutex> l(h->mtx);
        rc = body();
        ev.swap(h->deferred);
        cb = CallbackSet{h->sentence_cb, h->sentence_user, h->chars_cb, h->chars_user, h->ssdv_cb, h->ssdv_user, h->tracker, h->tracker_off};
    }
    if (!ev.empty()) fire_deferred(ev, cb);
    return rc;
}
} // namespace

static void fill_ssdv_info(hbd_ssdv_packet_info& info, const SsdvEvent& ev)
{
    memset(&info, 0, sizeof(info));
    memcpy(info.callsign, ev.header.callsign, sizeof(info.callsign));
    info.image_id = ev.header.image_id; info.packet_id = ev.header.packet_id;
    info.width = ev.header.width; info.height = ev.header.height;
    info.errors = ev.errors; info.set_size = ev.set_size;
}

#define HBD_CHECK_H(h)  if (!(h)) return HBD_ERR_ARG
#define HBD_CHECK_CH(h, ch) if (!(h) || (ch) < 0 || (ch) >= (h)->n_ch) return HBD_ERR_ARG

int hbd_decoder::alloc_fixed()
{
    const size_t n = size_t(n_ch);
    HBD_CUDA_CHECK(dev_alloc(d_state, n));
    {
        ChanState init;
        fresh_state(init);
        std::vector<ChanState> all(n, init);
        HBD_CUDA_CHECK(cudaMemcpy(d_state.get(), all.data(), n * sizeof(ChanState), cudaMemcpyHostToDevice));
    }
    HBD_CUDA_CHECK(dev_alloc(d_plan, n));
    for (DevPtr<float2>& c : d_carry2) {
        HBD_CUDA_CHECK(dev_alloc(c, n * size_t(carry_cap)));
        HBD_CUDA_CHECK(cudaMemset(c.get(), 0, n * size_t(carry_cap) * sizeof(float2)));
    }
    { const int rc = make_fft(fft_n, fft); if (rc) return rc; }
    HBD_CUDA_CHECK(dev_alloc(d_uart_runs, n * size_t(kUartRunsCap)));
    HBD_CUDA_CHECK(dev_alloc(d_maskc, n * size_t(2 * kMaskWords)));
    HBD_CUDA_CHECK(dev_alloc(d_lptaps, n * kLpMaxTaps));
    HBD_CUDA_CHECK(cudaMemset(d_lptaps.get(), 0, n * kLpMaxTaps * sizeof(float)));
    // character log: at least 512 entries per channel (a 600 baud channel decodes ~2 characters per 65 536-sample call,
    // so that is > 250 calls between drains even when every channel is noise); log_pressure() drains before it fills
    log_cap = kLogCapMin;
    while (size_t(log_cap) < 512 * n && log_cap < (1u << 30)) log_cap <<= 1;
    HBD_CUDA_CHECK(dev_alloc(d_log, size_t(log_cap)));
    HBD_CUDA_CHECK(dev_alloc(d_log_ctl, size_t(kCtlWords)));
    HBD_CUDA_CHECK(cudaMemset(d_log_ctl.get(), 0, kCtlWords * sizeof(unsigned)));
    HBD_CUDA_CHECK(stream_create(copy_stream));
    ev_call.resize(kMaxCallsBetweenCollects * 2);
    for (Event& e : ev_call) HBD_CUDA_CHECK(event_create(e));
    HBD_CUDA_CHECK(host_alloc(h_heads, ev_call.size() * kCtlWords));
    memset(h_heads.get(), 0, ev_call.size() * kCtlWords * sizeof(unsigned));
    HBD_CUDA_CHECK(host_alloc(h_tail_pin, 2));
    call_chars.resize(n);
    HBD_CUDA_CHECK(dev_alloc(d_taps1, 512));
    HBD_CUDA_CHECK(dev_alloc(d_taps2, 512));
    HBD_CUDA_CHECK(dev_alloc(d_cfg_baud, n));
    HBD_CUDA_CHECK(dev_alloc(d_cfg_stops, n));
    HBD_CUDA_CHECK(dev_alloc(d_cfg_bits, n));
    HBD_CUDA_CHECK(dev_alloc(d_cfg_dc, n));
    HBD_CUDA_CHECK(dev_alloc(d_cfg_ntaps, n));
    HBD_CUDA_CHECK(dev_alloc(d_cfg_dirty, n));
    HBD_CUDA_CHECK(dev_alloc(d_nco, n));
    h_nco.resize(n);
    HBD_CUDA_CHECK(dev_alloc(d_dacc_n, n));
    HBD_CUDA_CHECK(cudaMemset(d_dacc_n.get(), 0, n * sizeof(unsigned)));
    HBD_CUDA_CHECK(dev_alloc(d_frame_sizes, n));
    h_frame_sizes.resize(n);
    return HBD_OK;
}

// spectrum buffers + twiddle table of an N-point spectrum into `f` (hbd_create, hbd_set_fft_size)
int hbd_decoder::make_fft(int N_, FftBufs& f)
{
    const size_t n = size_t(n_ch), N = size_t(N_);
    HBD_CUDA_CHECK(dev_alloc(f.buf, n * N));
    HBD_CUDA_CHECK(cudaMemset(f.buf.get(), 0, n * N * sizeof(float2)));
    HBD_CUDA_CHECK(dev_alloc(f.spectrum, n * N));
    HBD_CUDA_CHECK(cudaMemset(f.spectrum.get(), 0, n * N * sizeof(float2)));
    HBD_CUDA_CHECK(dev_alloc(f.power, n * N));
    HBD_CUDA_CHECK(cudaMemset(f.power.get(), 0, n * N * sizeof(float)));
    // [0, N): exp(-2 pi i e / N); behind it the twiddles of the 4096-point (sub-)transform in the order its threads read
    // them: pass 1 [k1][t] = W_4096^(t k1) (16 x 256), pass 2 [j1][m2] = W_256^(m2 j1) (16 x 16); all evaluated in float64
    HBD_CUDA_CHECK(dev_alloc(f.twiddle, N + 4096 + 256));
    std::vector<float2> tw(N + 4096 + 256);
    auto w = [](double num, double den) { const double ang = -2.0 * M_PI * num / den; return make_float2(float(std::cos(ang)), float(std::sin(ang))); };
    for (size_t e = 0; e < N; ++e) tw[e] = w(double(e), double(N));
    for (size_t k1 = 0; k1 < 16; ++k1) for (size_t t = 0; t < 256; ++t) tw[N + k1 * 256 + t] = w(double(t * k1), 4096.0);
    for (size_t j1 = 0; j1 < 16; ++j1) for (size_t m2 = 0; m2 < 16; ++m2) tw[N + 4096 + j1 * 16 + m2] = w(double(16 * m2 * j1), 4096.0);
    HBD_CUDA_CHECK(cudaMemcpy(f.twiddle.get(), tw.data(), sizeof(float2) * tw.size(), cudaMemcpyHostToDevice));
    return HBD_OK;
}

// Install a decimation plan (a list of (M, taps) stages with the given total factor): K1 runs stages[0], the tail kernel the
// last stage, mid.cu the ones in between.  A new plan starts from fresh decimators (Decoder.h:283-284,347-348:
// decimation_stages_.clear()); unconsumed input stays queued (iq_in_buffer_ is untouched) -- it sits at the end of the carry.
// Taps and carry of the new plan go into locals first: on failure the previous plan stays in force.
int hbd_decoder::set_plan(const std::vector<TapTable>& st, size_t total_factor)
{
    if (settle()) return HBD_ERR_CUDA;
    const size_t n = size_t(n_ch);
    sync_ctrs();
    const TapTable none{1, nullptr, 1};   // M == 1: no such stage (a plan without one keeps the tap buffer it has)
    const TapTable &first = st.empty() ? none : st[0], &last = st.size() >= 2 ? st.back() : none;
    auto upload = [](DevPtr<float>& d, const TapTable& t, size_t cap) {
        cudaError_t e = t.bits ? dev_alloc(d, cap) : cudaSuccess;
        if (e == cudaSuccess && t.bits) e = cudaMemcpy(d.get(), t.bits, 4 * size_t(t.len), cudaMemcpyHostToDevice);
        return e;
    };
    DevPtr<float> taps1, taps2;
    HBD_CUDA_CHECK(upload(taps1, first, 512));
    HBD_CUDA_CHECK(upload(taps2, last, 512));
    std::vector<MidStage> new_mids;
    unsigned div = unsigned(first.M);
    for (size_t k = 1; k + 1 < st.size(); ++k) {
        MidStage m;
        m.M = st[k].M; m.T = st[k].len; m.div_in = div;
        HBD_CUDA_CHECK(upload(m.d_taps, st[k], size_t(m.T)));
        new_mids.push_back(std::move(m));
        div *= unsigned(st[k].M);
    }
    // the carry holds T1-1 samples of history plus the unconsumed remainder (< total factor).  Fresh, zeroed rows (new
    // decimators have an empty history); the remainder queued under the old plan stays queued, as in the reference
    unsigned max_r = 0;
    for (const auto& x : hc) max_r = std::max(max_r, x.in_r);
    const int cap = std::max(kCarryCapMin, int((size_t(first.len) + std::max<size_t>(total_factor, max_r) + 64 + 63) & ~size_t(63)));
    DevPtr<float2> fresh[2];
    for (DevPtr<float2>& f : fresh) {
        HBD_CUDA_CHECK(dev_alloc(f, n * size_t(cap)));
        HBD_CUDA_CHECK(cudaMemset(f.get(), 0, n * size_t(cap) * sizeof(float2)));
    }
    for (size_t c = 0; c < n; ++c)
        if (hc[c].in_r)
            HBD_CUDA_CHECK(cudaMemcpy(fresh[carry_cur].get() + c * size_t(cap) + size_t(cap) - hc[c].in_r,
                                      d_carry2[carry_cur].get() + c * size_t(carry_cap) + size_t(carry_cap) - hc[c].in_r, sizeof(float2) * hc[c].in_r,
                                      cudaMemcpyDeviceToDevice));
    for (int i = 0; i < 2; ++i) if (s1x.get(i)) HBD_CUDA_CHECK(cudaMemset(s1x.get(i), 0, n * s1x.pitch * sizeof(float2)));
    // commit
    factor = int(total_factor);
    M1 = first.M; T1 = first.len; M2 = last.M; T2 = last.len;
    if (taps1) d_taps1 = std::move(taps1);
    if (taps2) d_taps2 = std::move(taps2);
    mids = std::move(new_mids);
    midlast = {};
    carry_cap = cap;
    for (int i = 0; i < 2; ++i) d_carry2[i] = std::move(fresh[i]);
    for (auto& x : hc) { x.grown1 = x.grown2 = 0; for (size_t& g : x.grown_mid) g = 0; }
    cap_n_in = 0;
    h_plan_uploaded.clear();
    baud_fs = 0;   // fs_dec (the histograms' unit) may have changed, and the stream starts over
    return HBD_OK;
}

// size the per-call buffers for pushes of up to n_in_max (carried + new) samples per channel.  Every matrix that grows is
// filled into a local first; they are swapped in together once all of them are ready.
int hbd_decoder::ensure_call_capacity(size_t n_in_max)
{
    if (n_in_max <= cap_n_in && s1x.get()) return HBD_OK;
    const size_t n = size_t(n_ch);
    const size_t grow_to = std::max(n_in_max, cap_n_in);
    const size_t n1_max = grow_to / size_t(M1) + 2, n2_max = grow_to / size_t(factor) + 2;
    bool grown = false;
    auto regrow = [&](const auto& cur, auto& next, size_t width, size_t keep) {
        const cudaError_t e = cur.regrow(next, (width + 15) & ~size_t(15), n, keep, stream);
        grown = grown || next.p[0];
        return e;
    };
    Rows<float2, 2> s1, ml, rc;
    std::vector<Rows<float2>> mo(mids.size());
    Rows<float2> dq; Rows<float> sl, dm;
    HBD_CUDA_CHECK(regrow(s1x, s1, kS1Hist + n1_max, kS1Hist));
    for (size_t k = 0; k < mids.size(); ++k) {   // cascaded plan: the buffers between the stages
        const size_t n_out_max = grow_to / (size_t(mids[k].div_in) * size_t(mids[k].M)) + 2;
        if (k + 1 < mids.size()) HBD_CUDA_CHECK(regrow(mids[k].out, mo[k], kMidHist + n_out_max, kMidHist));
        else HBD_CUDA_CHECK(regrow(midlast, ml, kS1Hist + n_out_max, kS1Hist));
    }
    HBD_CUDA_CHECK(regrow(decq, dq, kLpHist + kLpBatch + n2_max, kLpHist + kLpBatch));
    HBD_CUDA_CHECK(regrow(slicer, sl, size_t(kSlicerVent) + 1 + kLpBatch + n2_max, slicer.pitch));
    HBD_CUDA_CHECK(regrow(demod, dm, kLpBatch + n2_max, 0));
    DevPtr<unsigned char> bits; DevPtr<unsigned> bits_n;
    if (record) {
        HBD_CUDA_CHECK(regrow(rec, rc, kLpBatch + n2_max, 0));
        if (!d_rec_bits) {
            HBD_CUDA_CHECK(dev_alloc(bits, n * (size_t(1) << 16)));
            HBD_CUDA_CHECK(dev_alloc(bits_n, n));
            HBD_CUDA_CHECK(cudaMemset(bits_n.get(), 0, n * sizeof(unsigned)));
        }
    }
    if (grown) HBD_CUDA_CHECK(cudaStreamSynchronize(stream));
    s1x.commit(s1);
    for (size_t k = 0; k < mids.size(); ++k) mids[k].out.commit(mo[k]);
    midlast.commit(ml);
    decq.commit(dq); slicer.commit(sl); demod.commit(dm); rec.commit(rc);
    if (bits) { d_rec_bits = std::move(bits); d_rec_bits_n = std::move(bits_n); rec_bits_pitch = 1u << 16; }
    cap_n_in = grow_to;
    return HBD_OK;
}

// No CUDA calls in here.  Returns HBD_OK or HBD_ERR_ARG (nothing has been changed in that case)
static int step_channel(hbd_decoder* h, HostChan& x, unsigned pushed, ChanStep& o, std::vector<float>& taps)
{
    const int factor = h->factor, M1 = h->M1, T1 = h->T1, M2 = h->M2, T2 = h->T2;
    const double fs_dec = h->fs_in / factor;
    ChanPlan& p = o.plan;
    p.r = x.in_r; p.n = pushed;
    p.dec_pending = x.dec_pending; p.lp_ntaps = unsigned(x.lp_ntaps);
    const unsigned total = x.in_r + pushed;
    if (int(total) < factor) {            // Decoder.h:429-430
        p.consumed = 0; p.n1 = p.n2 = 0; p.flags = 1;
        x.in_r = total; x.pushed = 0; x.last_n2 = 0; x.last_nf = 0;
        return HBD_OK;
    }
    p.consumed = total - total % unsigned(factor);
    p.n1 = p.consumed / unsigned(M1);
    p.n2 = p.consumed / unsigned(factor);
    p.flags = 0;
    // ---- everything that can fail comes first: the low-pass design (pure) --------------------------------
    const unsigned total_dec = x.dec_pending + p.n2;
    const bool gated = total_dec < unsigned(kLpBatch);                 // Decoder.h:494-495
    const bool cut_off = !gated && fs_dec > 4 * 40e3;                  // Decoder.h:522-527
    unsigned nf = 0;
    size_t T = x.lp_ntaps;
    bool redesign = false;
    if (!gated && !cut_off) {
        nf = total_dec - total_dec % unsigned(kLpBatch);
        const bool dirty = x.lp_dirty || x.lp_input_size != nf;
        if (dirty) {                                                   // Decoder.h:536-538
            T = design_lowpass(float(x.lp_bw / fs_dec), x.lp_trans, nf, x.lp_ntaps, taps);
            if (T > size_t(kLpMaxTaps)) { h->set_error("low-pass needs more than kLpMaxTaps (1025) taps: raise lowpass_trans"); return HBD_ERR_ARG; }
            redesign = T != x.lp_ntaps;
        }
    }
    // ---- commit ----------------------------------------------------------------------------------------------
    x.in_r = total - p.consumed;
    x.pushed = 0;
    x.last_n2 = p.n2; x.last_nf = 0;
    if (M1 > 1) {   // history re-zeroing when the reference's work buffers grow (Decimator.h:74-79)
        const size_t need = size_t(p.consumed) + size_t(T1) + size_t(M1);
        if (x.grown1 < need) { x.grown1 = need; o.zero_carry = true; }
    }
    size_t n_in = p.n1;            // samples entering the next stage
    for (size_t k = 0; k < h->mids.size(); ++k) {
        const size_t need = n_in + size_t(h->mids[k].T) + size_t(h->mids[k].M);
        if (x.grown_mid[k] < need) { x.grown_mid[k] = need; o.zero_mid |= 1u << k; }
        n_in /= size_t(h->mids[k].M);
    }
    if (M2 > 1) {
        const size_t need = n_in + size_t(T2) + size_t(M2);
        if (x.grown2 < need) { x.grown2 = need; o.zero_s1hist = true; }
    }
    if (gated) { x.dec_pending = total_dec; return HBD_OK; }
    if (cut_off) { x.dec_pending = 0; return HBD_OK; }
    x.dec_pending = total_dec - nf;
    x.last_nf = nf; x.demod_n = nf; o.nf = nf;
    x.lp_input_size = nf; x.lp_dirty = false;
    if (redesign) {
        o.taps_changed = true; o.taps_old = x.lp_ntaps; o.taps_new = T;
        x.lp_ntaps = T; h->derived_dirty = true;
    }
    p.lp_ntaps = unsigned(x.lp_ntaps);
    const size_t need = size_t(nf) + x.lp_ntaps;
    if (x.grown_lp < need) { x.grown_lp = need; o.zero_lphist = true; }   // FirFilter.h:141-147
    return HBD_OK;
}

// FFT frame assembly, Decoder.h:467-473 (mirror of K2's arithmetic): a frame fill `have` after n2 more decimated samples;
// true when the call completes the frame (K4 transforms it and clears the fill in that call)
static bool step_frame(unsigned& have, unsigned n2, unsigned fft_n)
{
    if (!n2 || have >= fft_n) return false;
    have += std::min(fft_n - have, n2);
    if (have < fft_n) return false;
    have = 0;
    return true;
}

// Keep the character / SSDV logs from filling up: look at what the completed calls have appended (their committed
// heads sit in pinned host memory, so this costs an event query, not a copy) and drain early when the calls still in
// flight could exhaust the space that is left.
int hbd_decoder::log_pressure()
{
    while (done_seq != call_seq && cudaEventQuery(ev_call[done_seq % ev_call.size()].get()) == cudaSuccess) {
        const unsigned head = h_heads.get()[size_t(done_seq % ev_call.size()) * kCtlWords + kCtlCharHead];
        per_call_max = std::max(per_call_max, head - done_head);
        done_head = head;
        ++done_seq;
    }
    const unsigned in_flight = call_seq - done_seq + 1u;     // the call about to be enqueued included
    const unsigned long long worst = (unsigned long long)(done_head - log_tail) + 2ull * in_flight * std::max(per_call_max, unsigned(n_ch));
    bool drain = worst > log_cap;
    if (ssdv_on && done_seq) {
        const unsigned sh = h_heads.get()[size_t((done_seq - 1u) % ev_call.size()) * kCtlWords + kCtlSsdvHead];
        if (sh - ssdv_log_tail > kSsdvLogCap / 2u) drain = true;
    }
    if (call_seq - calls_collected >= ev_call.size() / 2u) drain = true;   // event / head slots are about to be reused
    if (!drain || call_seq == calls_collected) return HBD_OK;
    return collect_locked(call_seq - calls_collected > 2u ? 1u : 0u);
}

// One ChanStep's side effects on the rows [c0, c0 + rows) of the per-channel buffers: a uniform call applies channel 0's
// step to every row (0, n_ch), a per-channel call each channel's step to its own row (c, 1).
int hbd_decoder::apply_step(const ChanStep& st, size_t c0, size_t rows, const std::vector<float>& taps)
{
    if (!(st.zero_carry || st.zero_s1hist || st.zero_mid || st.zero_lphist || st.taps_changed)) return HBD_OK;
    if (quiesce()) return HBD_ERR_CUDA;
    auto zero = [&](float2* p, size_t pitch, size_t w) {   // w samples from p on, in each of the rows of a [n_ch][pitch] matrix
        return cudaMemset2DAsync(p + c0 * pitch, pitch * sizeof(float2), 0, w * sizeof(float2), rows, stream);
    };
    if (st.zero_carry) HBD_CUDA_CHECK(zero(d_carry2[carry_cur].get() + (carry_cap - (T1 - 1) - int(st.plan.r)), size_t(carry_cap), size_t(T1 - 1)));
    for (size_t k = 0; k < mids.size(); ++k)
        if (st.zero_mid & (1u << k)) { const StageRows s = stage_in(k); HBD_CUDA_CHECK(zero(s.p, s.pitch, size_t(s.hist))); }
    if (st.zero_s1hist) { const StageRows s = stage_in(mids.size()); HBD_CUDA_CHECK(zero(s.p, s.pitch, size_t(s.hist))); }
    if (st.taps_changed) {
        std::vector<float> all(rows * st.taps_new);
        for (size_t c = 0; c < rows; ++c) memcpy(all.data() + c * st.taps_new, taps.data(), 4 * st.taps_new);
        HBD_CUDA_CHECK(cudaMemcpy2DAsync(d_lptaps.get() + c0 * kLpMaxTaps, kLpMaxTaps * sizeof(float), all.data(), st.taps_new * sizeof(float), st.taps_new * sizeof(float), rows,
                                         cudaMemcpyHostToDevice, stream));
        HBD_CUDA_CHECK(cudaStreamSynchronize(stream)); // `all` goes out of scope
        for (size_t c = c0; c < c0 + rows; ++c) hc[c].cfg_dirty = true;   // lp_ntaps travels with the configuration upload
        cfg_dirty_any = true;
    }
    if (st.zero_lphist) HBD_CUDA_CHECK(zero(decq.get(), decq.pitch, std::min<size_t>(st.plan.lp_ntaps, kLpHist)));
    return HBD_OK;
}

// The host half of a process call: step the counters of the channels (channel 0 alone in uniform mode), size the per-call
// buffers, apply the side effects, upload configuration and plans.  Everything in a call that may wait for the GPU is here.
int hbd_decoder::plan_call(CallPlan& cp)
{
    const size_t n = size_t(n_ch);
    groups_idle = false;
    // uniform mode (whole-batch pushes only, one low-pass setting): channel 0 stands for all of them, O(1) per call
    const bool uni = ctr_uniform && lp_cfg_uniform;
    if (!uni) { leave_uniform(); h_plan.resize(n); }
    const size_t stepped = uni ? 1 : n;
    auto pushed = [&](size_t c) { return in.p ? unsigned(in.n) : hc[c].pushed; };
    size_t max_total = 0;
    for (size_t c = 0; c < stepped; ++c) max_total = std::max<size_t>(max_total, size_t(hc[c].in_r) + pushed(c));
    if (max_total > cap_n_in || !s1x.get()) { if (quiesce()) return HBD_ERR_CUDA; }   // buffers are about to be reallocated
    { const int rc = ensure_call_capacity(max_total); if (rc) return rc; }
    if (baud_on) { const int rc = baud_start(); if (rc) return rc; }
    unsigned max_nf = 0;
    std::vector<float> new_taps;
    for (size_t c = 0; c < stepped; ++c) {
        ChanStep st;
        int rc = step_channel(this, hc[c], pushed(c), st, new_taps);
        if (rc) return rc;   // channels below c have been stepped: their samples are gone (documented in the header)
        if (uni) { ctr_stale = true; cp.uplan = st.plan; } else { h_plan[c] = st.plan; cp.need_k4 |= step_frame(hc[c].fft_have, st.plan.n2, unsigned(fft_n)); }
        cp.any_work |= !(st.plan.flags & 1u);
        cp.max_n1 = std::max(cp.max_n1, st.plan.n1); max_nf = std::max(max_nf, st.nf);
        rc = apply_step(st, c, uni ? n : 1, new_taps);
        if (rc) return rc;
    }
    if (uni) {   // each frame level once; levels that complete their frames in the same call are all back at 0: merge them
        unsigned done = 0;
        for (unsigned& v : fft_lvl) done += step_frame(v, cp.uplan.n2, unsigned(fft_n)) ? 1u : 0u;
        cp.need_k4 = done > 0;
        plan_steps += unsigned(fft_lvl.size());
        if (done > 1) {
            std::vector<unsigned> to(fft_lvl.size()), merged;
            for (size_t i = 0; i < fft_lvl.size(); ++i) {
                to[i] = unsigned(std::find(merged.begin(), merged.end(), fft_lvl[i]) - merged.begin());
                if (to[i] == merged.size()) merged.push_back(fft_lvl[i]);
            }
            for (unsigned& l : lvl_of) l = to[l];
            fft_lvl.swap(merged);
        }
    } else plan_steps += unsigned(n);
    if (demod_acc_on) { const int rc = ensure_dacc(); if (rc) return rc; }

    if (cfg_dirty_any) {
        if (quiesce()) return HBD_ERR_CUDA;
        sync_ctrs();
        std::vector<double> b(n); std::vector<float> s(n); std::vector<int> bi(n), dc(n), nt(n); std::vector<unsigned char> d(n);
        for (size_t c = 0; c < n; ++c) {
            b[c] = hc[c].baud; s[c] = hc[c].rtty_stops; bi[c] = int(hc[c].rtty_bits); dc[c] = hc[c].dc_remove; nt[c] = int(hc[c].lp_ntaps);
            d[c] = hc[c].cfg_dirty; hc[c].cfg_dirty = false;
        }
        HBD_CUDA_CHECK(cudaMemcpyAsync(d_cfg_baud.get(), b.data(), 8 * n, cudaMemcpyHostToDevice, stream));
        HBD_CUDA_CHECK(cudaMemcpyAsync(d_cfg_stops.get(), s.data(), 4 * n, cudaMemcpyHostToDevice, stream));
        HBD_CUDA_CHECK(cudaMemcpyAsync(d_cfg_bits.get(), bi.data(), 4 * n, cudaMemcpyHostToDevice, stream));
        HBD_CUDA_CHECK(cudaMemcpyAsync(d_cfg_dc.get(), dc.data(), 4 * n, cudaMemcpyHostToDevice, stream));
        HBD_CUDA_CHECK(cudaMemcpyAsync(d_cfg_ntaps.get(), nt.data(), 4 * n, cudaMemcpyHostToDevice, stream));
        HBD_CUDA_CHECK(cudaMemcpyAsync(d_cfg_dirty.get(), d.data(), n, cudaMemcpyHostToDevice, stream));
        init_cfg_kernel<<<(n_ch + 127) / 128, 128, 0, stream>>>(d_state.get(), d_cfg_baud.get(), d_cfg_stops.get(), d_cfg_bits.get(), d_cfg_dc.get(), d_cfg_ntaps.get(), d_cfg_dirty.get(), n_ch);
        ++launches;
        HBD_CUDA_CHECK(cudaStreamSynchronize(stream)); // host vectors go out of scope
        cfg_dirty_any = false;
    }
    if (!uni) {
        // back to uniform mode as soon as the channels agree again (e.g. after a round of per-channel pushes of one size)
        regroup();
        for (size_t c = 1; c < n && cp.plan_uniform; ++c) cp.plan_uniform = memcmp(&h_plan[c], &h_plan[0], sizeof(ChanPlan)) == 0;
        cp.uplan = h_plan[0];
        if (!cp.plan_uniform && (h_plan_uploaded.size() != n || memcmp(h_plan.data(), h_plan_uploaded.data(), n * sizeof(ChanPlan)) != 0)) {
            if (quiesce()) return HBD_ERR_CUDA;
            HBD_CUDA_CHECK(cudaMemcpyAsync(d_plan.get(), h_plan.data(), n * sizeof(ChanPlan), cudaMemcpyHostToDevice, stream));
            HBD_CUDA_CHECK(cudaStreamSynchronize(stream));
            h_plan_uploaded = h_plan;
        }
    }

    // what the tail kernel stages in shared memory: sized from host-side knowledge of all channels
    if (derived_dirty) {
        sync_ctrs();
        const double fs_dec = fs_in / factor;
        max_lp_taps_c = 1; max_spb_c = 1;
        for (size_t c = 0; c < n; ++c) {
            max_lp_taps_c = std::max(max_lp_taps_c, hc[c].lp_ntaps);
            if (hc[c].baud > 0) max_spb_c = std::max(max_spb_c, fs_dec / hc[c].baud);
        }
        derived_dirty = false;
    }
    // a channel normally holds < ~12 symbols of pending samples after a slicer pass (plus this call's batch)
    cp.sv_want = int(std::min<double>(6144.0, 16.0 * max_spb_c + double(max_nf) + 64.0));
    if (sv_override >= 0) cp.sv_want = sv_override;   // test hook (HBD_SV_WANT): 0 forces the slicer's HBM path
    return HBD_OK;
}

// The device half of a process call: the kernel sequence on the hi / lo streams, the commit of the log heads and the
// ping-pong flips.  No allocation, no synchronisation.
int hbd_decoder::enqueue_call(const CallPlan& cp)
{
    const double fs_dec = fs_in / factor;
    const float2* chunk = in.p ? static_cast<const float2*>(in.p) : stage.get();
    const size_t chunk_pitch = in.p ? in.pitch : stage.pitch;
    int nl = 0;
    // everything the caller (and the host-side updates of plan_call) put on `stream` happens before the kernels start
    HBD_CUDA_CHECK(cudaEventRecord(ev_in.get(), stream));
    HBD_CUDA_CHECK(cudaStreamWaitEvent(hi.get(), ev_in.get(), 0));
    bool tail_recorded = false;
    // K1 overwrites the stage-1 buffer: the tail of the call before the previous one must be done with it
    if (tail_pending[s1_cur]) HBD_CUDA_CHECK(cudaStreamWaitEvent(hi.get(), ev_tail[s1_cur].get(), 0));
    {   // K1 also writes the next call's carry (even when no channel has a full decimation block yet)
        DecimArgs da{};
        da.chunk = chunk; da.chunk_pitch = chunk_pitch; da.carry = d_carry2[carry_cur].get(); da.carry_next = d_carry2[carry_cur ^ 1].get(); da.carry_cap = carry_cap;
        da.s1 = s1x.get(s1_cur); da.s1_pitch = s1x.pitch; da.s1_hist = kS1Hist;
        da.plan = d_plan.get(); da.uplan = cp.uplan; da.uniform = cp.plan_uniform ? 1 : 0; da.taps = d_taps1.get(); da.ch0 = 0; da.n_channels = n_ch;
        da.nco = in.nco;
        if (timing) HBD_CUDA_CHECK(cudaEventRecord(next_event(ev_k1, ev_used_k1), hi.get()));
        HBD_CUDA_CHECK(launch_decim1(da, M1, T1, cp.max_n1, n_sms, hi.get(), &nl, in.format));
        if (timing) HBD_CUDA_CHECK(cudaEventRecord(next_event(ev_k1, ev_used_k1), hi.get()));
    }
    HBD_CUDA_CHECK(cudaEventRecord(ev_consumed.get(), hi.get())); // input no longer needed; stage-1 output ready
    HBD_CUDA_CHECK(cudaStreamWaitEvent(lo.get(), ev_consumed.get(), 0));
    if (timing > 1) HBD_CUDA_CHECK(cudaEventRecord(next_event(ev_rest, ev_used_rest), lo.get()));
    if (cp.any_work) {
        // cascaded plan: the stages between K1's and the tail kernel's (1/64 of the input rate or less)
        for (size_t k = 0; k < mids.size(); ++k) {
            const StageRows in_k = stage_in(k), out_k = stage_in(k + 1);
            MidArgs ma{};
            ma.plan = d_plan.get(); ma.uplan = cp.uplan; ma.uniform = cp.plan_uniform ? 1 : 0;
            ma.in = in_k.p; ma.in_next = in_k.next; ma.in_pitch = in_k.pitch; ma.in_hist = in_k.hist;
            ma.out = out_k.p; ma.out_pitch = out_k.pitch; ma.out_hist = out_k.hist;
            ma.taps = mids[k].d_taps.get(); ma.M = mids[k].M; ma.T = mids[k].T; ma.div_in = mids[k].div_in;
            HBD_CUDA_CHECK(launch_mid_stage(ma, n_ch, lo.get(), &nl));
        }
        const StageRows s1 = stage_in(mids.size());
        TailArgs ta{};
        ta.plan = d_plan.get(); ta.uplan = cp.uplan; ta.uniform = cp.plan_uniform ? 1 : 0; ta.state = d_state.get(); ta.ch0 = 0;
        ta.s1 = s1.p; ta.s1_next = s1.next; ta.s1_pitch = s1.pitch;
        ta.taps2 = d_taps2.get(); ta.M2 = M2; ta.T2 = T2;
        ta.decq = decq.get(); ta.dq_pitch = decq.pitch; ta.fs_dec = fs_dec; ta.fftbuf = fft.buf.get(); ta.fft_n = fft_n; ta.lptaps = d_lptaps.get();
        ta.max_lp_taps = int(max_lp_taps_c);
        ta.slicer = slicer.get(); ta.slicer_pitch = slicer.pitch; ta.sv_want = cp.sv_want;
        ta.log = d_log.get(); ta.log_ctl = d_log_ctl.get(); ta.log_mask = log_cap - 1u; ta.call_seq = call_seq & 0xffffffu;
        ta.uart_runs = d_uart_runs.get();
        ta.maskc = mask_cache ? d_maskc.get() : nullptr;
        ta.ssdv_ring = ssdv_on ? d_ssdv_ring.get() : nullptr; ta.ssdv_total = d_ssdv_total.get();
        ta.demod_last = demod.get(); ta.demod_pitch = demod.pitch;
        ta.rec_decimated = record ? rec.get(0) : nullptr; ta.rec_filtered = record ? rec.get(1) : nullptr; ta.rec_pitch = rec.pitch;
        ta.rec_bits = record ? d_rec_bits.get() : nullptr; ta.rec_bits_n = d_rec_bits_n.get(); ta.rec_bits_pitch = rec_bits_pitch;
        HBD_CUDA_CHECK(launch_tail(ta, n_ch, lo.get(), &nl));
        // only the tail kernel reads the stage-1 buffer: K1 of the call after next may overwrite it as soon as the
        // tail is done, without waiting for the FFT / SSDV / demod kernels behind it on this stream
        if (!tail_ev_late) { HBD_CUDA_CHECK(cudaEventRecord(ev_tail[s1_cur].get(), lo.get())); tail_recorded = true; }
        if (baud_on) {   // the run histograms, from the discriminator output the tail kernel has just written
            BaudHistArgs ba{};
            ba.plan = d_plan.get(); ba.uplan = cp.uplan; ba.uniform = cp.plan_uniform ? 1 : 0; ba.state = d_state.get();
            ba.demod = demod.get(); ba.demod_pitch = demod.pitch;
            ba.hist = d_bhist.get(); ba.hist_pitch = size_t(baud_lmax) + 1; ba.track = d_btrack.get();
            const BaudGeometry g = baud_geometry(fs_dec);
            ba.lmax = g.lmax; ba.m = g.m;
            HBD_CUDA_CHECK(launch_baud_hist(ba, n_ch, lo.get(), &nl));
        }
        FftArgs fa{};
        fa.state = d_state.get(); fa.fftbuf = fft.buf.get(); fa.spectrum = fft.spectrum.get(); fa.power = fft.power.get(); fa.twiddle = fft.twiddle.get(); fa.fs_dec = fs_dec;
        fa.ch0 = 0; fa.fft_n = fft_n;
        if (cp.need_k4) HBD_CUDA_CHECK(launch_fft_afc(fa, n_ch, lo.get(), &nl));   // other calls: K2 has stepped the AFC itself
        if (ssdv_on) {   // test every 0x55-started window the new characters completed
            SsdvScanArgs sa{};
            sa.ring = d_ssdv_ring.get(); sa.total = d_ssdv_total.get(); sa.scanned = d_ssdv_scanned.get(); sa.log = d_ssdv_log.get();
            sa.ctl = d_log_ctl.get(); sa.call_seq = call_seq & 0xffffffu; sa.ch0 = 0;
            HBD_CUDA_CHECK(launch_ssdv_scan(sa, n_ch, lo.get(), &nl));
        }
    }
    if (demod_acc_on && demod.get()) { // main.cpp:267-282 runs after EVERY process(), also when nothing new was demodulated
        DemodAccArgs aa{};
        aa.state = d_state.get(); aa.demod = demod.get(); aa.demod_pitch = demod.pitch; aa.acc = dacc.get(); aa.acc_pitch = dacc.pitch; aa.acc_n = d_dacc_n.get();
        aa.fs_dec = fs_dec; aa.ch0 = 0;
        HBD_CUDA_CHECK(launch_demod_accumulate(aa, n_ch, lo.get(), &nl));
    }
    if (timing > 1) HBD_CUDA_CHECK(cudaEventRecord(next_event(ev_rest, ev_used_rest), lo.get()));
    if (!tail_recorded) HBD_CUDA_CHECK(cudaEventRecord(ev_tail[s1_cur].get(), lo.get()));
    tail_pending[s1_cur] = true;
    // the caller's stream resumes once the input has been consumed (it does not wait for the tail kernels)
    HBD_CUDA_CHECK(cudaStreamWaitEvent(stream, ev_consumed.get(), 0));
    carry_cur ^= 1;
    if (cp.any_work) s1_cur ^= 1; // the tail (which moves the stage-2 history to the other buffer) ran
    launches += unsigned(nl);
    if (snap_on) {
        stats_snap_kernel<<<(n_ch + 127) / 128, 128, 0, lo.get()>>>(d_state.get(), d_snap.get() + size_t(call_seq % kSnapSlots) * size_t(n_ch) * 6, n_ch);
        ++launches;
    }
    // commit: the log control words as they stand after this call, into the call's pinned slot (stream order: every
    // entry below these heads is completely written when ev_call fires)
    const size_t slot = call_seq % ev_call.size();
    HBD_CUDA_CHECK(cudaMemcpyAsync(h_heads.get() + slot * kCtlWords, d_log_ctl.get(), kCtlWords * sizeof(unsigned), cudaMemcpyDeviceToHost, lo.get()));
    HBD_CUDA_CHECK(cudaEventRecord(ev_call[slot].get(), lo.get())); // everything of this call is done
    ++call_seq;
    return HBD_OK;
}

int hbd_decoder::process_async_locked()
{
    if (!fs_in) return HBD_OK; // Decoder.h:418-419: uninitialised -> silently nothing
    HBD_CUDA_CHECK(cudaSetDevice(device));
    { const int rc = log_pressure(); if (rc) return rc; }
    CallPlan cp;
    const auto t_plan0 = std::chrono::steady_clock::now();
    { const int rc = plan_call(cp); if (rc) return rc; }
    plan_host_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_plan0).count();
    if (in.p && in.format != HBD_IQ_CF32 && !decim1_supports_native_iq(M1, T1)) {   // the plan changed after a native integer push
        size_t wp = 0;
        const int rc = widen(in.p, in.pitch, in.format, n_ch, in.n, &wp);
        if (rc) return rc;
        in = DeviceInput{d_widen(), wp, in.n};
    }
    { const int rc = enqueue_call(cp); if (rc) return rc; }
    in = DeviceInput{};
    return HBD_OK;
}

// entries [tail, tail + n) of a device ring of `cap` entries (a power of two) into dst: one copy, or two where the range
// wraps, then a synchronise of `s` (none for n == 0)
template <class T>
static cudaError_t read_ring(std::vector<T>& dst, const T* ring, unsigned cap, unsigned tail, unsigned n, cudaStream_t s)
{
    dst.resize(n);
    if (!n) return cudaSuccess;
    const unsigned i0 = tail & (cap - 1u), first = std::min(n, cap - i0);
    cudaError_t e = cudaMemcpyAsync(dst.data(), ring + i0, size_t(first) * sizeof(T), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess && n > first) e = cudaMemcpyAsync(dst.data() + first, ring, size_t(n - first) * sizeof(T), cudaMemcpyDeviceToHost, s);
    return e == cudaSuccess ? cudaStreamSynchronize(s) : e;
}

// Drain decoded characters of all calls up to (last enqueued - lag) and run the sentence layer on them, call by
// call like Decoder::process().  lag == 0 waits for everything; lag > 0 leaves the newest calls in flight so the GPU
// keeps working while the host is busy here.  User callbacks are only RECORDED here (h->deferred).
int hbd_decoder::collect_locked(unsigned lag)
{
    HBD_CUDA_CHECK(cudaSetDevice(device));
    if (call_seq == calls_collected) return lag == 0 ? settle() : HBD_OK;
    if (call_seq - calls_collected <= lag) return HBD_OK;
    if (lag == 0 && call_seq - calls_collected > 2) {
        // a full drain behind a queue of calls: take the finished calls first, in halving steps, so the host's sentence
        // layer works while the GPU is still busy with the newest calls instead of after it has gone idle
        int first_rc = HBD_OK;
        for (unsigned l = (call_seq - calls_collected) / 2; l >= 1; l /= 2) { const int rc = collect_locked(l); if (rc == HBD_ERR_CUDA) return rc; if (rc && !first_rc) first_rc = rc; }
        const int rc = collect_locked(0);
        return rc ? rc : first_rc;
    }
    const unsigned upto = call_seq - lag;            // calls [calls_collected, upto) get drained
    if (lag == 0) {
        if (settle()) return HBD_ERR_CUDA;
    } else {
        HBD_CUDA_CHECK(cudaEventSynchronize(ev_call[(upto - 1) % ev_call.size()].get()));
    }
    // the COMMITTED control words of call upto-1 (never the live head: newer calls may be appending right now)
    unsigned heads[kCtlWords];
    memcpy(heads, h_heads.get() + size_t((upto - 1) % ev_call.size()) * kCtlWords, sizeof(heads));
    const unsigned head = heads[kCtlCharHead];
    int result = HBD_OK;
    if (ssdv_on) {
        // accepted SSDV packets of the calls being drained go to their channels first: the buffer automaton below
        // looks a window's verdict up when it reaches it, which is never before the call that completed the window
        // the overflow words are monotonic counters: a change since the previous drain is reported once, decoding goes on
        if (heads[kCtlSsdvRingOvf] != ovf_seen[0]) {
            ovf_seen[0] = heads[kCtlSsdvRingOvf];
            set_error("SSDV character ring overflow: more than 3840 characters in one call (windows lost); push smaller chunks");
            result = HBD_ERR_STATE;
        }
        if (heads[kCtlSsdvOvf] != ovf_seen[1]) {
            set_error("SSDV packet log overflow: " + std::to_string(heads[kCtlSsdvOvf] - ovf_seen[1]) + " packet(s) lost; collect more often");
            ovf_seen[1] = heads[kCtlSsdvOvf];
            result = HBD_ERR_STATE;
        }
        HBD_CUDA_CHECK(read_ring(h_ssdv_log, d_ssdv_log.get(), kSsdvLogCap, ssdv_log_tail, std::min(heads[kCtlSsdvHead] - ssdv_log_tail, kSsdvLogCap),
                                 copy_stream.get()));
        for (const SsdvLogEntry& e : h_ssdv_log) {
            if (e.ch >= unsigned(n_ch)) continue;
            SsdvVerdict v; v.pos = e.pos; v.errors = e.errors; memcpy(v.data.data(), e.data, 256);
            ssdv[e.ch].verdicts.push_back(v);
        }
        ssdv_log_tail = heads[kCtlSsdvHead];
    }
    if (heads[kCtlCharOvf] != ovf_seen[2]) {
        // a writer found the ring full and dropped its characters (it never overwrites unread entries).  Which slots of
        // the range were skipped is not recorded, so the whole range is given up; decoding continues behind it.
        ovf_seen[2] = heads[kCtlCharOvf];
        chars_lost += head - log_tail;
        set_error("decoded-character log overflow: " + std::to_string(head - log_tail) + " characters of calls [" + std::to_string(calls_collected) + ", " +
                  std::to_string(upto) + ") lost; collect more often");
        log_tail = head;
        result = HBD_ERR_STATE;
    }
    if (snap_on && call_seq - (upto - 1u) < kSnapSlots - 1u) {   // the slot of call upto-1 has not been reused yet
        HBD_CUDA_CHECK(cudaMemcpyAsync(h_snap.get(), d_snap.get() + size_t((upto - 1u) % kSnapSlots) * size_t(n_ch) * 6, sizeof(float) * 6 * size_t(n_ch),
                                       cudaMemcpyDeviceToHost, copy_stream.get()));
        h_snap_valid = true;
    }
    HBD_CUDA_CHECK(read_ring(h_log, d_log.get(), log_cap, log_tail, head - log_tail, copy_stream.get()));
    // the writers may reuse everything below the new tail
    log_tail = head;
    h_tail_pin.get()[0] = log_tail; h_tail_pin.get()[1] = ssdv_log_tail;
    HBD_CUDA_CHECK(cudaMemcpyAsync(d_log_ctl.get() + kCtlCharTail, h_tail_pin.get(), sizeof(unsigned), cudaMemcpyHostToDevice, copy_stream.get()));
    HBD_CUDA_CHECK(cudaMemcpyAsync(d_log_ctl.get() + kCtlSsdvTail, h_tail_pin.get() + 1, sizeof(unsigned), cudaMemcpyHostToDevice, copy_stream.get()));
    HBD_CUDA_CHECK(cudaStreamSynchronize(copy_stream.get()));   // h_tail_pin is rewritten by the next drain

    // The log is sorted by call, and within a call a channel's characters form ONE contiguous segment (one reservation per
    // flush; only a channel that decodes more than kCharBuf = 64 characters in a call flushes twice).  Replay segment by
    // segment: one TextChannel::feed per channel and call, like one Decoder::process().
    const auto t_replay0 = std::chrono::steady_clock::now();
    const size_t n_log = h_log.size();
    seg_start.clear();
    for (size_t i = 0; i < n_log;) {           // segment boundaries: one sequential pass over the copied log
        size_t j = i + 1;
        while (j < n_log && h_log[j].x == h_log[i].x && (h_log[j].y >> 8) == (h_log[i].y >> 8)) ++j;
        seg_start.push_back(unsigned(i));
        i = j;
    }
    seg_start.push_back(unsigned(n_log));
    const size_t n_seg = seg_start.size() - 1;
    // Channels are independent, so the replay is cut by CHANNEL RANGE over a few host threads (the caller's included):
    // every thread walks all segments in log order and takes the ones of its channels -- per channel the order of the
    // calls is kept, and the callbacks the threads record are merged back into log order afterwards.
    const bool want_sent = sentence_cb || tracker;
    int n_thr = std::max(1, std::min(host_threads, int(n_seg / 1024)));
    n_thr = std::min(n_thr, n_ch);
    std::vector<ReplayPart> parts;
    parts.resize(size_t(n_thr));
    auto replay = [&](int t) {
        ReplayPart& part = parts[size_t(t)];
        const int c_lo = int((long long)n_ch * t / n_thr), c_hi = int((long long)n_ch * (t + 1) / n_thr);
        unsigned cur_seg = 0;
        SentenceSink sink;
        if (want_sent)
            sink = [&part, &cur_seg](int ch, const std::string& cs, const std::string& d, const std::string& crc) {
                Deferred ev; ev.kind = Deferred::kSentence; ev.ch = ch; ev.a = cs; ev.b = d; ev.c = crc;
                part.events.emplace_back(cur_seg, std::move(ev));
            };
        auto feed_channel = [&](int ch, const unsigned char* chars, size_t n_chars) {
            TextChannel& tc = text[size_t(ch)];
            hbd_result_record& pr = pend[size_t(ch)];
            const size_t before = chars_cb ? tc.chars_size(pr) : 0;
            tc.feed(chars, n_chars, ch, sink, keep_raw, pr);
            if (!tc.chars_spill.empty() || !tc.sent_spill.empty()) part.spilled = true;
            if (chars_cb && tc.chars_size(pr) > before) {   // character_callback_, Decoder.h:617-629 (not paced by wall clock)
                Deferred ev; ev.kind = Deferred::kChars; ev.ch = ch; ev.a = tc.chars_from(pr, before);
                part.events.emplace_back(cur_seg, std::move(ev));
            }
            if (ssdv_on) {   // Decoder.h:573: one SSDV_wraper_t::push per call that decoded characters
                SsdvEvent sev;
                if (ssdv[size_t(ch)].push(chars, n_chars, sev)) {
                    ssdv[size_t(ch)].events_pending.push_back(sev);
                    if (ssdv_cb) {   // ssdv_callback_, Decoder.h:631-632
                        Deferred ev; ev.kind = Deferred::kSsdv; ev.ch = ch; fill_ssdv_info(ev.info, sev); ev.pkt = sev.data;
                        part.events.emplace_back(cur_seg, std::move(ev));
                    }
                }
            }
        };
        std::vector<int> split;                    // channels of this range whose characters of the current call span several segments
        unsigned char seg_chars[kCharBufHost];
        // the per-channel state is scattered over the heap: a short look-ahead queue of this range's next segments feeds prefetches
        size_t look = 0;
        unsigned ahead[8]; int n_ahead = 0, head = 0;
        auto refill = [&] {
            while (n_ahead < 8 && look < n_seg) {
                const unsigned c = h_log[seg_start[look]].x;
                if (c >= unsigned(c_lo) && c < unsigned(c_hi)) {
                    ahead[(head + n_ahead) & 7] = unsigned(look); ++n_ahead;
                    __builtin_prefetch(&text[c]); __builtin_prefetch(&pend[c]);
                }
                ++look;
            }
        };
        refill();
        while (n_ahead) {
            const size_t k = ahead[head]; head = (head + 1) & 7; --n_ahead;
            refill();
            if (n_ahead >= 4) text[h_log[seg_start[ahead[(head + 3) & 7]]].x].prefetch_tails();
            cur_seg = unsigned(k);
            const size_t i0 = seg_start[k], i1 = seg_start[k + 1];
            const int ch = int(h_log[i0].x);
            const unsigned seq = h_log[i0].y >> 8;
            const size_t len = i1 - i0;
            // a full buffer means the channel flushed more than once in this call: join the pieces (rare: > 64 characters of
            // one channel in one call); they need not be adjacent in the log
            bool joined = len >= size_t(kCharBufHost);
            if (!joined && !split.empty()) joined = std::find(split.begin(), split.end(), ch) != split.end();
            if (joined) {
                if (call_chars[size_t(ch)].empty()) split.push_back(ch);
                for (size_t i = i0; i < i1; ++i) call_chars[size_t(ch)].push_back(char(h_log[i].y & 0xffu));
            } else {
                for (size_t i = 0; i < len; ++i) seg_chars[i] = (unsigned char)(h_log[i0 + i].y & 0xffu);
                feed_channel(ch, seg_chars, len);
            }
            // end of this call's entries (for this range): feed the joined channels
            if (!split.empty() && (!n_ahead || (h_log[seg_start[ahead[head]]].y >> 8) != seq)) {
                for (int sc : split) {
                    std::string& cc = call_chars[size_t(sc)];
                    feed_channel(sc, reinterpret_cast<const unsigned char*>(cc.data()), cc.size());
                    cc.clear();
                }
                split.clear();
            }
        }
    };
    pool.run(n_thr, replay);     // part t on worker t (it finds its channels' text state in its cache), late workers' parts on this thread
    {   // callbacks back into log order (stable: a channel's events keep the order they were recorded in)
        size_t total = 0;
        for (const ReplayPart& pt : parts) { total += pt.events.size(); if (pt.spilled) spill_free = false; }
        if (total) {
            std::vector<std::pair<unsigned, Deferred>> all;
            all.reserve(total);
            for (ReplayPart& pt : parts) for (auto& e : pt.events) all.push_back(std::move(e));
            if (n_thr > 1) std::stable_sort(all.begin(), all.end(), [](const auto& x, const auto& y) { return x.first < y.first; });
            for (auto& e : all) deferred.push_back(std::move(e.second));
        }
    }
    drain_host_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_replay0).count();
    drain_calls += upto - calls_collected;
    calls_collected = upto;
    return result;
}

// SSDV packet sync on / off.  Switching it on starts from an empty character stream (like a freshly constructed
// SSDV_wraper_t): every call in flight is drained first, so device ring, scan position and host automaton agree.
int hbd_decoder::enable_ssdv(bool on)
{
    if (on == ssdv_on) return HBD_OK;
    HBD_CUDA_CHECK(cudaSetDevice(device));
    { const int rc = collect_locked(0); if (rc) return rc; }
    const size_t n = size_t(n_ch);
    if (on) {
        if (!d_ssdv_ring) {   // the four buffers are allocated together
            DevPtr<unsigned char> ring; DevPtr<unsigned> total, scanned; DevPtr<SsdvLogEntry> log;
            HBD_CUDA_CHECK(dev_alloc(ring, n * kSsdvRing));
            HBD_CUDA_CHECK(dev_alloc(total, n));
            HBD_CUDA_CHECK(dev_alloc(scanned, n));
            HBD_CUDA_CHECK(dev_alloc(log, size_t(kSsdvLogCap)));
            d_ssdv_ring = std::move(ring); d_ssdv_total = std::move(total); d_ssdv_scanned = std::move(scanned); d_ssdv_log = std::move(log);
        }
        HBD_CUDA_CHECK(cudaMemset(d_ssdv_ring.get(), 0, n * kSsdvRing));
        HBD_CUDA_CHECK(cudaMemset(d_ssdv_total.get(), 0, n * sizeof(unsigned)));
        HBD_CUDA_CHECK(cudaMemset(d_ssdv_scanned.get(), 0, n * sizeof(unsigned)));
        // the SSDV log keeps its (monotonic) head: nothing below it is of interest any more
        ssdv_log_tail = h_heads.get()[size_t((call_seq ? call_seq - 1u : 0u) % ev_call.size()) * kCtlWords + kCtlSsdvHead];
        h_tail_pin.get()[1] = ssdv_log_tail;
        HBD_CUDA_CHECK(cudaMemcpy(d_log_ctl.get() + kCtlSsdvTail, h_tail_pin.get() + 1, sizeof(unsigned), cudaMemcpyHostToDevice));
        ssdv.assign(n, SsdvChannel());
    }
    ssdv_on = on;
    return HBD_OK;
}

int hbd_decoder::enable_snap()
{
    if (snap_on) return HBD_OK;
    HBD_CUDA_CHECK(cudaSetDevice(device));
    if (!d_snap) {   // both buffers are allocated together
        DevPtr<float> d; HostPtr<float> hp;
        HBD_CUDA_CHECK(dev_alloc(d, size_t(kSnapSlots) * size_t(n_ch) * 6));
        HBD_CUDA_CHECK(cudaMemset(d.get(), 0, sizeof(float) * size_t(kSnapSlots) * size_t(n_ch) * 6));
        HBD_CUDA_CHECK(host_alloc(hp, 6 * size_t(n_ch)));
        memset(hp.get(), 0, sizeof(float) * 6 * size_t(n_ch));
        d_snap = std::move(d); h_snap = std::move(hp);
    }
    snap_on = true;
    return HBD_OK;
}

// hbd_reset_channels: the listed channels become channel 0 of a new handle with the same settings.  The drain comes first,
// so that what the calls in flight decoded goes through the old text and SSDV state; then the host state restarts and one
// kernel restarts the device state on the handle's stream (the next call's K1 waits for it through ev_in).
int hbd_decoder::reset_channels(const int* chs, size_t k)
{
    std::vector<unsigned char> listed(size_t(n_ch), 0);
    for (size_t i = 0; i < k; ++i) {
        if (chs[i] < 0 || chs[i] >= n_ch || listed[size_t(chs[i])]) { set_error("reset_channels: channel out of range or listed twice"); return HBD_ERR_ARG; }
        listed[size_t(chs[i])] = 1;
    }
    if (!k) return HBD_OK;
    sync_ctrs();
    bool staged = in.p != nullptr;
    for (size_t c = 0; c < hc.size() && !staged; ++c) staged = hc[c].pushed != 0;
    if (staged) { set_error("reset_channels: pushed samples have not been processed yet"); return HBD_ERR_STATE; }
    HBD_CUDA_CHECK(cudaSetDevice(device));
    { const int rc = collect_locked(0); if (rc) return rc; }   // also: the previous reset's list upload is complete
    if (!h_reset) {   // both buffers are allocated together
        HostPtr<int> hp; DevPtr<int> dp;
        HBD_CUDA_CHECK(host_alloc(hp, size_t(n_ch)));
        HBD_CUDA_CHECK(dev_alloc(dp, size_t(n_ch)));
        h_reset = std::move(hp); d_reset = std::move(dp);
    }
    leave_uniform();
    for (size_t i = 0; i < k; ++i) {
        const size_t c = size_t(chs[i]);
        HostChan& x = hc[c];
        x.ctr() = ChanCtr();   // grown* == 0: the next call zeroes the carry and stage histories of this row (apply_step)
        x.fft_have = 0; x.nco_phase = 0;
        x.cfg_dirty = true;    // the configuration goes onto the fresh ChanState with the next call's upload, as on a new handle
        text[c].restart();
        if (c < ssdv.size()) ssdv[c].restart();
        h_reset.get()[i] = chs[i];
    }
    cfg_dirty_any = derived_dirty = true;
    regroup();   // resetting every channel keeps the handle uniform, on one frame level
    HBD_CUDA_CHECK(cudaMemcpyAsync(d_reset.get(), h_reset.get(), k * sizeof(int), cudaMemcpyHostToDevice, stream));
    ResetArgs a{};
    a.state = d_state.get(); a.list = d_reset.get();
    a.decq = decq.get(); a.dq_pitch = decq.pitch;
    a.dacc_n = d_dacc_n.get(); a.ssdv_total = d_ssdv_total.get(); a.ssdv_scanned = d_ssdv_scanned.get(); a.rec_bits_n = d_rec_bits_n.get();
    a.bhist = d_bhist.get(); a.bhist_pitch = size_t(baud_lmax) + 1; a.btrack = d_btrack.get();
    reset_chan_kernel<<<unsigned(k), 128, 0, stream>>>(a);
    ++launches;
    HBD_CUDA_CHECK(cudaGetLastError());
    return HBD_OK;
}

// (Re)start every channel's baud estimator for the current fs_dec: rows sized for its histogram, zeroed.  A no-op while
// the rows are current; otherwise it waits for the compute streams.  A failed allocation changes nothing.
int hbd_decoder::baud_start()
{
    const double fs = fs_in / factor;
    if (baud_fs == fs) return HBD_OK;
    const size_t n = size_t(n_ch);
    const BaudGeometry g = baud_geometry(fs);
    const size_t pitch = size_t(g.lmax) + 1;
    if (sync_groups()) { set_error("stream sync failed"); return HBD_ERR_CUDA; }   // a histogram kernel may still use the rows
    DevPtr<unsigned> hist; DevPtr<BaudTrack> track; DevPtr<hbd_baud_estimate> est;
    if (!d_bhist || g.lmax != baud_lmax) {   // the three buffers are allocated together
        if (dev_alloc(hist, n * pitch) != cudaSuccess || dev_alloc(track, n) != cudaSuccess || dev_alloc(est, n) != cudaSuccess) {
            set_error("baud estimation: out of device memory");
            return HBD_ERR_NOMEM;
        }
    }
    HBD_CUDA_CHECK(cudaMemsetAsync(hist ? hist.get() : d_bhist.get(), 0, n * pitch * sizeof(unsigned), stream));
    HBD_CUDA_CHECK(cudaMemsetAsync(track ? track.get() : d_btrack.get(), 0, n * sizeof(BaudTrack), stream));
    HBD_CUDA_CHECK(cudaStreamSynchronize(stream));
    if (hist) { d_bhist = std::move(hist); d_btrack = std::move(track); d_best = std::move(est); baud_lmax = g.lmax; }
    baud_fs = fs;
    return HBD_OK;
}

// every channel's estimate as of all calls enqueued so far (estimation on): zeros before the first push, else one score
// kernel once everything enqueued is done, and one copy
int hbd_decoder::baud_estimates(std::vector<hbd_baud_estimate>& out)
{
    out.assign(size_t(n_ch), hbd_baud_estimate{});
    if (!fs_in) return HBD_OK;
    HBD_CUDA_CHECK(cudaSetDevice(device));
    { const int rc = baud_start(); if (rc) return rc; }
    if (settle()) return HBD_ERR_CUDA;
    HBD_CUDA_CHECK(launch_baud_score(d_bhist.get(), size_t(baud_lmax) + 1, baud_lmax, d_btrack.get(), fs_in / factor, d_best.get(), n_ch, stream));
    ++launches;
    HBD_CUDA_CHECK(cudaMemcpyAsync(out.data(), d_best.get(), out.size() * sizeof(hbd_baud_estimate), cudaMemcpyDeviceToHost, stream));
    HBD_CUDA_CHECK(cudaStreamSynchronize(stream));
    return HBD_OK;
}

namespace hbd {
int internal_device(hbd_decoder* h) { return h->device; }
void internal_set_error(hbd_decoder* h, const std::string& what) { std::lock_guard<std::mutex> l(h->mtx); h->set_error(what); }
DistSlot& internal_dist_slot(hbd_decoder* h) { return h->dist_ctx; }
}

// =====================================================================================================
extern "C" {

// One record per channel with what the sentence layer has produced since the previous pack (printable characters, CRC-valid
// sentences; what does not fit a record stays for the next one) and the AFC scalars as of the newest drained call.
size_t hbd_pack_results(hbd_decoder* h, int ch_offset, hbd_result_record* out, size_t cap_records)
{
    if (!h) return 0;
    std::lock_guard<std::mutex> l(h->mtx);
    const size_t n = size_t(h->n_ch);
    if (!out || cap_records < n) return n;
    std::vector<float> live;     // AFC scalars when no snapshot has been taken yet
    const float* st = h->h_snap.get();
    if (!(h->snap_on && h->h_snap_valid)) {   // read the live state (waits for the calls in flight)
        if (h->enable_snap() != HBD_OK) return 0;
        std::vector<ChanState> cs(n);
        if (h->read_states(0, n, cs.data())) return 0;
        live.resize(6 * n);
        for (size_t c = 0; c < n; ++c) afc_scalars(cs[c], live.data() + 6 * c);
        st = live.data();
    }
    // the pending slots ARE the records: copy, stamp, reset (and move spilled bytes up).  Cut by channel range like the
    // replay of the drain, so that a range is packed by the thread that filled it.
    const bool spill_free = h->spill_free;
    const int n_thr = int(std::max<size_t>(1, std::min<size_t>(size_t(h->host_threads), n / 1024)));
    std::vector<unsigned char> left(size_t(n_thr), 0);
    h->pool.run(n_thr, [&](int t) {
        const size_t c_lo = n * size_t(t) / size_t(n_thr), c_hi = n * size_t(t + 1) / size_t(n_thr);
        bool any_left = false;
        for (size_t c = c_lo; c < c_hi; ++c) {
            hbd_result_record& pr = h->pend[c];
            hbd_result_record& o = out[c];
            // header + the bytes in use only (the rest of a record is not read by anybody)
            o.n_chars = pr.n_chars; o.sentence_bytes = pr.sentence_bytes; o.reserved = 0;
            if (pr.n_chars) memcpy(o.chars, pr.chars, pr.n_chars);
            if (pr.sentence_bytes) memcpy(o.sentences, pr.sentences, pr.sentence_bytes);
            o.channel = uint32_t(ch_offset + int(c));
            const float* sc = st + 6 * c;
            o.frequency_correction = sc[0]; o.shift = sc[1]; o.noise_floor = sc[2]; o.noise_variance = sc[3];
            o.peak_left = int32_t(sc[4]); o.peak_right = int32_t(sc[5]);
            o.n_sentences = pr.sentence_bytes ? uint16_t(std::count(pr.sentences, pr.sentences + pr.sentence_bytes, '\n')) : uint16_t(0);
            pr.n_chars = 0; pr.sentence_bytes = 0;
            uint16_t fl = 0;
            if (__builtin_expect(!spill_free, 0)) {
                TextChannel& tc = h->text[c];
                if (!tc.chars_spill.empty()) { fl |= 1u; TextChannel::refill(pr.chars, pr.n_chars, sizeof(pr.chars), tc.chars_spill); }
                if (!tc.sent_spill.empty()) { fl |= 2u; TextChannel::refill(pr.sentences, pr.sentence_bytes, sizeof(pr.sentences), tc.sent_spill); }
                any_left = any_left || !tc.chars_spill.empty() || !tc.sent_spill.empty();
            }
            o.flags = fl;
        }
        left[size_t(t)] = any_left;
    });
    if (!h->spill_free) h->spill_free = std::find(left.begin(), left.end(), 1) == left.end();
    return n;
}
int hbd_set_stats_snapshot(hbd_decoder* h, int on)
{
    HBD_CHECK_H(h);
    std::lock_guard<std::mutex> l(h->mtx);
    if (on) return h->enable_snap();
    h->snap_on = false; h->h_snap_valid = false;
    return HBD_OK;
}

int hbd_create(int n_channels, int cuda_device, hbd_decoder** out)
{
    if (!out || n_channels < 1) return HBD_ERR_ARG;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || cuda_device < 0 || cuda_device >= count) return HBD_ERR_CUDA;
    if (cudaSetDevice(cuda_device) != cudaSuccess) return HBD_ERR_CUDA;
    std::unique_ptr<hbd_decoder> h(new (std::nothrow) hbd_decoder);
    if (!h) return HBD_ERR_NOMEM;
    h->n_ch = n_channels; h->device = cuda_device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, cuda_device) == cudaSuccess) h->n_sms = prop.multiProcessorCount;
    h->hc.resize(size_t(n_channels));
    h->lvl_of.assign(size_t(n_channels), 0u);
    h->text.resize(size_t(n_channels));
    for (auto& tc : h->text) { tc.text_stream.reserve(120); tc.last_sentence.reserve(96); }   // no allocation on the drain path in steady state
    { hbd_result_record z; memset(&z, 0, sizeof(z)); h->pend.assign(size_t(n_channels), z); }
    if (stream_create(h->own_stream) != cudaSuccess) return HBD_ERR_CUDA;
    h->stream = h->own_stream.get();
    {
        if (const char* sv = getenv("HBD_SV_WANT")) h->sv_override = atoi(sv);
        if (const char* mc = getenv("HBD_MASK_CACHE")) h->mask_cache = atoi(mc) != 0;
        if (const char* tl = getenv("HBD_TAIL_EV_LATE")) h->tail_ev_late = atoi(tl) != 0;
        if (const char* nf = getenv("HBD_NCO_FUSED")) h->nco_fused = atoi(nf) != 0;
        {
            cpu_set_t set;
            int cores = int(std::thread::hardware_concurrency());
            if (sched_getaffinity(0, sizeof(set), &set) == 0) cores = CPU_COUNT(&set);
            h->host_threads = std::max(1, std::min(4, cores / 2));   // measured on 8 ranks x 4 cores: 2 threads 0.44 ms/step, 4 threads 0.51 (stalls)
            if (const char* ht = getenv("HBD_HOST_THREADS")) h->host_threads = std::max(1, atoi(ht));
        }
        int prio_lo = 0, prio_hi = 0;
        cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi); // numerically lower = higher priority
        if (stream_create(h->hi, prio_hi) != cudaSuccess || stream_create(h->lo, prio_lo) != cudaSuccess) return HBD_ERR_CUDA;
        if (event_create(h->ev_consumed) != cudaSuccess || event_create(h->ev_tail[0]) != cudaSuccess || event_create(h->ev_tail[1]) != cudaSuccess ||
            event_create(h->ev_in) != cudaSuccess) return HBD_ERR_CUDA;
    }
    const int rc = h->alloc_fixed();
    if (rc) return rc;
    *out = h.release();
    return HBD_OK;
}

void hbd_destroy(hbd_decoder* h) { delete h; }

const char* hbd_last_error(hbd_decoder* h) { return h ? h->err.c_str() : "null handle"; }

int hbd_set_stream(hbd_decoder* h, void* s)
{
    HBD_CHECK_H(h);
    std::lock_guard<std::mutex> l(h->mtx);
    if (h->settle()) return HBD_ERR_CUDA;
    h->own_stream.reset();
    h->stream = (cudaStream_t)s;
    return HBD_OK;
}

// 4096 (the reference's fft_bins_cnt_) or 16384; restarts spectrum collection and the AFC of every channel
int hbd_set_fft_size(hbd_decoder* h, size_t n_bins)
{
    HBD_CHECK_H(h);
    if (n_bins != size_t(kFftN) && n_bins != size_t(kFftNMax)) return HBD_ERR_ARG;
    std::lock_guard<std::mutex> l(h->mtx);
    if (h->settle()) return HBD_ERR_CUDA;
    if (int(n_bins) == h->fft_n) return HBD_OK;
    hbd_decoder::FftBufs f;   // swapped in after the state reset below: on failure the old size and spectra stay
    const int rc = h->make_fft(int(n_bins), f);
    if (rc) return rc;
    // spectrum / AFC state back to a freshly constructed decoder's (Average<T> starts with one 0 sample)
    std::vector<ChanState> st(size_t(h->n_ch));
    if (h->read_states(0, st.size(), st.data())) return HBD_ERR_CUDA;
    for (auto& s : st) {
        s.fft_have = s.fft_ready = s.have_spectrum = 0;
        s.afc_correction = s.afc_noise_floor = s.afc_noise_var = s.afc_shift_hz = 0;
        s.nf_sum = s.nv_sum = 0; s.pl_sum = s.pr_sum = 0; s.nf_cnt = s.nv_cnt = s.pl_cnt = s.pr_cnt = 1;
        s.gui_left = s.gui_right = 0; s.spec_ok = 0;
    }
    if (cudaMemcpy(h->d_state.get(), st.data(), st.size() * sizeof(ChanState), cudaMemcpyHostToDevice) != cudaSuccess) return HBD_ERR_CUDA;
    h->fft = std::move(f);
    h->fft_n = int(n_bins);
    for (auto& x : h->hc) x.fft_have = 0;
    h->fft_lvl.assign(1, 0u);
    h->lvl_of.assign(h->hc.size(), 0u);
    return HBD_OK;
}

int hbd_set_record(hbd_decoder* h, int on)
{
    HBD_CHECK_H(h);
    std::lock_guard<std::mutex> l(h->mtx);
    h->record = on != 0;
    h->cap_n_in = 0; // force (re)allocation of the recording buffers on the next call
    return HBD_OK;
}

#define HBD_SETTER(NAME, TYPE, FIELD)                                                \
    int hbd_set_##NAME(hbd_decoder* h, int ch, TYPE v)                               \
    {                                                                                \
        if (!h || ch < -1 || ch >= h->n_ch) return HBD_ERR_ARG;                      \
        std::lock_guard<std::mutex> l(h->mtx);                                       \
        for (int c = (ch < 0 ? 0 : ch); c < (ch < 0 ? h->n_ch : ch + 1); ++c) {      \
            h->hc[size_t(c)].FIELD = v;                                              \
            h->hc[size_t(c)].cfg_dirty = true;                                       \
        }                                                                            \
        h->cfg_dirty_any = h->derived_dirty = true;                                  \
        return HBD_OK;                                                               \
    }
HBD_SETTER(baud, double, baud)
HBD_SETTER(rtty_bits, size_t, rtty_bits)
HBD_SETTER(rtty_stops, float, rtty_stops)
HBD_SETTER(dc_remove, int, dc_remove)

// Decoder::lowpass_bw / lowpass_trans re-run the design immediately (Decoder.h:238-257)
static int set_lp(hbd_decoder* h, int ch, float bw, float trans, bool set_bw)
{
    if (!h || ch < -1 || ch >= h->n_ch) return HBD_ERR_ARG;
    std::lock_guard<std::mutex> l(h->mtx);
    // FirFilter::LP_BlackmanHarris takes (size_t)(4 / trans) taps (clipped to the block length); the tap rows hold kLpMaxTaps
    if (!set_bw && trans != 0.f && !(4.0f / trans <= float(kLpMaxTaps - 1))) {
        h->set_error("lowpass_trans below 4/1024 needs more than kLpMaxTaps (1025) low-pass taps");
        return HBD_ERR_ARG;
    }
    cudaSetDevice(h->device);
    h->sync_groups();
    h->leave_uniform();
    std::vector<float> taps;
    for (int c = (ch < 0 ? 0 : ch); c < (ch < 0 ? h->n_ch : ch + 1); ++c) {
        HostChan& x = h->hc[size_t(c)];
        if (set_bw) x.lp_bw = bw; else x.lp_trans = trans;
        x.lp_dirty = true;
        if (!h->fs_in) continue;
        const double fs_dec = h->fs_in / h->factor;
        const size_t T = design_lowpass(float(x.lp_bw / fs_dec), x.lp_trans, x.lp_input_size, x.lp_ntaps, taps);
        if (T != x.lp_ntaps && T <= size_t(kLpMaxTaps)) {
            x.lp_ntaps = T; x.cfg_dirty = true; h->cfg_dirty_any = h->derived_dirty = true;
            if (cudaMemcpy(h->d_lptaps.get() + size_t(c) * kLpMaxTaps, taps.data(), 4 * T, cudaMemcpyHostToDevice) != cudaSuccess) return HBD_ERR_CUDA;
        }
    }
    bool cfg_same = true;
    for (size_t c = 1; c < h->hc.size(); ++c) cfg_same = cfg_same && h->hc[c].lp_bw == h->hc[0].lp_bw && h->hc[c].lp_trans == h->hc[0].lp_trans;
    h->lp_cfg_uniform = cfg_same;
    h->regroup();
    return HBD_OK;
}
int hbd_set_lowpass_bw(hbd_decoder* h, int ch, float bw) { return set_lp(h, ch, bw, 0, true); }
int hbd_set_lowpass_trans(hbd_decoder* h, int ch, float tr) { return set_lp(h, ch, 0, tr, false); }

#define HBD_GETTER(NAME, TYPE, FIELD)                                                \
    TYPE hbd_get_##NAME(hbd_decoder* h, int ch)                                      \
    {                                                                                \
        if (!h || ch < 0 || ch >= h->n_ch) return 0;                                 \
        std::lock_guard<std::mutex> l(h->mtx);                                       \
        return h->hc[size_t(ch)].FIELD;                                              \
    }
HBD_GETTER(baud, double, baud)
HBD_GETTER(rtty_bits, size_t, rtty_bits)
HBD_GETTER(rtty_stops, float, rtty_stops)
HBD_GETTER(lowpass_bw, float, lp_bw)
HBD_GETTER(lowpass_trans, float, lp_trans)
HBD_GETTER(dc_remove, int, dc_remove)

size_t hbd_setup_decimation_factor(hbd_decoder* h, size_t factor)
{
    if (!h) return 0;
    std::lock_guard<std::mutex> l(h->mtx);
    if (factor < 1 || factor > 256) return size_t(h->factor);
    std::vector<TapTable> st;
    if (!plan_for_factor(factor, st)) { h->set_plan(st, 1); return 0; }   // Decoder.h:283-284,317-319: stages cleared, factor 1, returns 0
    return h->set_plan(st, factor) == HBD_OK ? factor : 0;
}

// Decoder::setupDecimationStagesBW (Decoder.h:336-412): while the rate is above the limit, divide by the smallest power of
// two below 256 that gets under it -- or by 256 when none does -- and append that factor's stages.  Limits far below the
// input rate therefore cascade several plans (20 MS/s -> 5 kHz: /256 then /16 = (64,348t)(4,139t)(8,54t)(2,69t)).
size_t hbd_setup_decimation_bw(hbd_decoder* h, double max_rate)
{
    if (!h) return 0;
    std::lock_guard<std::mutex> l(h->mtx);
    if (!h->fs_in) return 0;
    double rate = h->fs_in;
    size_t total = 1;
    std::vector<TapTable> plan, st;
    while (rate > max_rate) {
        int div;
        for (div = 2; div < 256; div *= 2) if (rate / div <= max_rate) break;
        rate /= div; total *= size_t(div);
        plan_for_factor(size_t(div), st);
        plan.insert(plan.end(), st.begin(), st.end());
        if (total > 65536 || plan.size() > size_t(kMaxMidStages + 2)) {
            h->set_error("setup_decimation_bw: more than 8 stages / a total factor above 65536 is not supported");
            return 0;
        }
    }
    return h->set_plan(plan, total) == HBD_OK ? total : 0;
}

// ---- input: the hbd_push_* entry points ---------------------------------------------------------------------------------
// NCO parameters of channels [c0, c0 + nc) for a push of n samples into out[0, nc), and the channels' phases advanced past
// the push.  k0_rotation: also the rotation over kNcoThreads samples that K0 steps by (K1's fused mixer does not use it).
void hbd_decoder::nco_params(NcoChan* out, int c0, int nc, size_t n, bool k0_rotation)
{
    for (int i = 0; i < nc; ++i) {
        HostChan& x = hc[size_t(c0 + i)];
        NcoChan& k = out[i];
        k.inc = x.nco_freq / fs_in;
        k.ph0 = x.nco_phase;
        const double a = -2.0 * M_PI * k.inc * double(kNcoThreads);
        k.step_re = k0_rotation ? std::cos(a) : 1.0;
        k.step_im = k0_rotation ? std::sin(a) : 0.0;
        const double ph = x.nco_phase + double(n) * k.inc;
        x.nco_phase = ph - std::floor(ph);
    }
}

// K0: mix `n` samples per channel of channels [c0, c0+nc) from src into the staging rows at dst_off and advance the
// channels' NCO phases.  src_pitch 0: one shared (wideband) row.  Integer src (format) is widened on the way; a channel
// without an offset is then a plain widening copy.  Returns once the stream has caught up.
int hbd_decoder::mix_into_stage(const void* src, size_t src_pitch, int c0, int nc, size_t dst_off, size_t n, int format)
{
    if (!n) return HBD_OK;
    nco_params(h_nco.data() + c0, c0, nc, n, true);
    HBD_CUDA_CHECK(cudaMemcpyAsync(d_nco.get() + c0, h_nco.data() + c0, sizeof(NcoChan) * size_t(nc), cudaMemcpyHostToDevice, stream));
    int nl = 0;
    HBD_CUDA_CHECK(launch_nco_mix(src, src_pitch, stage.get(), stage.pitch, dst_off, n, d_nco.get(), c0, nc, stream, &nl, format));
    launches += unsigned(nl);
    HBD_CUDA_CHECK(cudaStreamSynchronize(stream)); // h_nco is rewritten by the next push
    return HBD_OK;
}

// K0 without a mixer: `rows` rows of n samples of `format` (row pitch `pitch`) -> cf32 d_widen [rows][*out_pitch] (even
// pitch: 16-byte rows), on the stream.  Work put on the stream after a process call waits for that call's K1
// (process_async_locked), so d_widen is free again by then.
int hbd_decoder::widen(const void* src, size_t pitch, int format, int rows, size_t n, size_t* out_pitch)
{
    *out_pitch = (n + 1) & ~size_t(1);
    HBD_CUDA_CHECK(widen_buf.grow(std::max<size_t>(size_t(rows) * *out_pitch * sizeof(float2), 256), 1, 0, stream));
    int nl = 0;
    HBD_CUDA_CHECK(launch_nco_mix(src, pitch, d_widen(), *out_pitch, 0, n, nullptr, 0, rows, stream, &nl, format));
    launches += unsigned(nl);
    return HBD_OK;
}

// One push, whichever entry point it came through: check the arguments, then, under the mutex, the state; latch the rate
// and take the route that gets the samples to where K1 reads them.  `base`: samples already staged in the rows pushed to.
//
//   source                                condition                                  route
//   host cf32, channel / matrix           -                                          copy into staging at base; K0 in place if
//                                                                                    the channel's NCO is set (channel) / nco_any
//   host integers, channel / matrix       -                                          upload to iq_up; K0 widens (and mixes)
//                                                                                    into staging at base
//   device cf32 matrix                    no nco_any                                 zero copy
//   device integer matrix                 no nco_any, decim1_supports_native_iq      zero copy, K1 reads the integers
//   device integer matrix                 otherwise                                  K0 widens into d_widen, then the device
//                                                                                    cf32 route on d_widen
//   device cf32 matrix with nco_any, or   nco_fused, base == 0, n > 0, 16-byte       fused NCO: K1 mixes while it decimates (a
//   any wideband row (a host or integer   aligned, decim1_supports_fused_nco         host row synchronises before returning)
//   row lands in d_widen as cf32 first)   otherwise                                  K0 mixes into staging at base
int hbd_decoder::push(const PushSrc& s)
{
    const size_t bytes = size_t(iq_bytes(s.format)), n = s.n;
    const bool channel = s.shape == PushSrc::kChannel, device_matrix = s.device && s.shape == PushSrc::kMatrix;
    if (!bytes || (channel && (s.ch < 0 || s.ch >= n_ch)) || (!s.p && (n || device_matrix))) return HBD_ERR_ARG;
    if (s.shape == PushSrc::kMatrix && s.pitch < n) return HBD_ERR_ARG;
    if (device_matrix && ((s.pitch * bytes) % 16 || (reinterpret_cast<uintptr_t>(s.p) & 15))) return HBD_ERR_ARG;

    std::lock_guard<std::mutex> l(mtx);
    if (in.p) { set_error("device push pending"); return HBD_ERR_STATE; }
    HBD_CUDA_CHECK(cudaSetDevice(device));
    const bool zero_copy = device_matrix && !nco_any;   // K1 reads the caller's matrix (or its widened copy) in place
    unsigned base = 0;
    if (channel) {
        if (n_ch > 1) leave_uniform();   // per-channel feeding: the counters are stepped channel by channel from here on
        base = hc[size_t(s.ch)].pushed;
    } else if (!queue_depth_equal(base) || (zero_copy && base)) {
        set_error(s.shape == PushSrc::kRow ? "wideband push needs equal queue depth in all channels"
                  : zero_copy              ? "host push pending"
                                           : "batch push needs equal queue depth in all channels");
        return HBD_ERR_STATE;
    }
    if (!fs_in) fs_in = double(float(s.fs));   // Decoder::init(const float)
    auto ensure_stage = [&] {
        return stage.grow((std::max(size_t(base) + n, stage.pitch) + 15) & ~size_t(15), size_t(n_ch), stage.pitch, stream);
    };

    if (!s.device && s.shape != PushSrc::kRow) {   // host channel / matrix: into the staging rows
        const int c0 = channel ? s.ch : 0, rows = channel ? 1 : n_ch;
        const bool cf32 = s.format == HBD_IQ_CF32;
        HBD_CUDA_CHECK(ensure_stage());
        if (!cf32 && n) HBD_CUDA_CHECK(iq_up.grow(size_t(rows) * n * bytes, 1, 0, stream));
        void* dst = cf32 ? (void*)(stage.get() + size_t(c0) * stage.pitch + base) : (void*)iq_up.get();   // integers cross PCIe packed [rows][n]
        const size_t dst_pitch = cf32 ? stage.pitch * sizeof(float2) : n * bytes;
        if (n) HBD_CUDA_CHECK(cudaMemcpy2DAsync(dst, dst_pitch, s.p, (channel ? n : s.pitch) * bytes, n * bytes, size_t(rows), cudaMemcpyHostToDevice, stream));
        const bool mix = channel ? hc[size_t(c0)].nco_freq != 0 || hc[size_t(c0)].nco_phase != 0 : nco_any;
        int rc = HBD_OK;
        if (!cf32) rc = mix_into_stage(iq_up.get(), channel ? 0 : n, c0, rows, base, n, s.format);
        else if (mix) rc = mix_into_stage(stage.get() + base, stage.pitch, c0, rows, base, n);   // in place
        else HBD_CUDA_CHECK(cudaStreamSynchronize(stream));
        if (rc) return rc;   // either way the stream has caught up: the caller owns `p` again (Decoder.h:209-213 copies)
        if (channel) hc[size_t(c0)].pushed += unsigned(n); else add_pushed(unsigned(n));
        return HBD_OK;
    }

    const void* src = s.p;
    size_t pitch = s.pitch;   // 0 for a row
    if (s.shape == PushSrc::kRow && !(s.device && s.format == HBD_IQ_CF32)) {   // the row lands in d_widen as cf32
        const bool cf32 = s.format == HBD_IQ_CF32;
        if (!s.device && n) {   // upload: cf32 straight into d_widen, integers into iq_up
            Rows<unsigned char>& up = cf32 ? widen_buf : iq_up;
            HBD_CUDA_CHECK(up.grow(n * bytes, 1, 0, stream));
            HBD_CUDA_CHECK(cudaMemcpyAsync(up.get(), s.p, n * bytes, cudaMemcpyHostToDevice, stream));
            src = up.get();
        }
        if (!cf32) { size_t wp = 0; const int rc = widen(src, 0, s.format, 1, n, &wp); if (rc) return rc; }
        src = d_widen();
    }
    if (device_matrix && s.format != HBD_IQ_CF32) {
        if (zero_copy && decim1_supports_native_iq(M1, T1)) { in = DeviceInput{s.p, s.pitch, n, s.format}; return HBD_OK; }
        const int rc = widen(s.p, s.pitch, s.format, n_ch, n, &pitch);
        if (rc) return rc;
        src = d_widen();
    }
    if (zero_copy) { in = DeviceInput{src, pitch, n}; return HBD_OK; }
    if (nco_fused && base == 0 && n && decim1_supports_fused_nco(M1, T1) && !(reinterpret_cast<uintptr_t>(src) & 15)) {
        // the raw samples stay where they are and K1 mixes while it decimates (decim1.cu, DecimArgs::nco): no K0 launch, no
        // 8-byte write + 8-byte read per channel-sample through HBM.  The parameters go through a ring of pinned slots, so
        // the push does not wait for the GPU.
        if (!s.device) HBD_CUDA_CHECK(cudaStreamSynchronize(stream));   // the caller owns `p` again on return
        if (!h_nco_pin) {   // the ring's buffers and events are created together
            HostPtr<NcoChan> hp; DevPtr<NcoChan> dp; Event ev[kNcoSlots];
            HBD_CUDA_CHECK(host_alloc(hp, size_t(n_ch) * kNcoSlots));
            HBD_CUDA_CHECK(dev_alloc(dp, size_t(n_ch) * kNcoSlots));
            for (Event& e : ev) HBD_CUDA_CHECK(event_create(e));
            h_nco_pin = std::move(hp); d_nco_ring = std::move(dp);
            for (unsigned i = 0; i < kNcoSlots; ++i) ev_nco[i] = std::move(ev[i]);
        }
        const unsigned slot = nco_seq % kNcoSlots;
        if (nco_seq >= kNcoSlots) HBD_CUDA_CHECK(cudaEventSynchronize(ev_nco[slot].get()));   // the upload that last used this pinned slot (16 pushes ago)
        ++nco_seq;
        NcoChan* hp = h_nco_pin.get() + size_t(slot) * size_t(n_ch);
        NcoChan* dp = d_nco_ring.get() + size_t(slot) * size_t(n_ch);
        nco_params(hp, 0, n_ch, n, false);
        HBD_CUDA_CHECK(cudaMemcpyAsync(dp, hp, sizeof(NcoChan) * size_t(n_ch), cudaMemcpyHostToDevice, stream));
        HBD_CUDA_CHECK(cudaEventRecord(ev_nco[slot].get(), stream));
        in = DeviceInput{src, pitch, n, HBD_IQ_CF32, dp};
        return HBD_OK;
    }
    HBD_CUDA_CHECK(ensure_stage());
    const int rc = mix_into_stage(src, pitch, 0, n_ch, base, n);
    if (rc) return rc;
    add_pushed(unsigned(n));
    return HBD_OK;
}

int hbd_push_samples(hbd_decoder* h, int ch, const float* iq, size_t n, double fs)
{ return h ? h->push({iq, false, HBD_IQ_CF32, PushSrc::kChannel, ch, 0, n, fs}) : HBD_ERR_ARG; }
int hbd_push_samples_batch(hbd_decoder* h, const float* iq, size_t n, size_t pitch, double fs)
{ return h ? h->push({iq, false, HBD_IQ_CF32, PushSrc::kMatrix, 0, pitch, n, fs}) : HBD_ERR_ARG; }
int hbd_push_samples_device(hbd_decoder* h, const float* d_iq, size_t n, size_t pitch, double fs)
{ return h ? h->push({d_iq, true, HBD_IQ_CF32, PushSrc::kMatrix, 0, pitch, n, fs}) : HBD_ERR_ARG; }
int hbd_push_wideband(hbd_decoder* h, const float* iq, size_t n, double fs)
{ return h ? h->push({iq, false, HBD_IQ_CF32, PushSrc::kRow, 0, 0, n, fs}) : HBD_ERR_ARG; }
int hbd_push_wideband_device(hbd_decoder* h, const float* d_iq, size_t n, double fs)
{ return h ? h->push({d_iq, true, HBD_IQ_CF32, PushSrc::kRow, 0, 0, n, fs}) : HBD_ERR_ARG; }
int hbd_push_iq(hbd_decoder* h, int ch, const void* iq, int format, size_t n, double fs)
{ return h ? h->push({iq, false, format, PushSrc::kChannel, ch, 0, n, fs}) : HBD_ERR_ARG; }
int hbd_push_iq_batch(hbd_decoder* h, const void* iq, int format, size_t n, size_t pitch, double fs)
{ return h ? h->push({iq, false, format, PushSrc::kMatrix, 0, pitch, n, fs}) : HBD_ERR_ARG; }
int hbd_push_iq_device(hbd_decoder* h, const void* d_iq, int format, size_t n, size_t pitch, double fs)
{ return h ? h->push({d_iq, true, format, PushSrc::kMatrix, 0, pitch, n, fs}) : HBD_ERR_ARG; }
int hbd_push_iq_wideband(hbd_decoder* h, const void* iq, int format, size_t n, double fs)
{ return h ? h->push({iq, false, format, PushSrc::kRow, 0, 0, n, fs}) : HBD_ERR_ARG; }
int hbd_push_iq_wideband_device(hbd_decoder* h, const void* d_iq, int format, size_t n, double fs)
{ return h ? h->push({d_iq, true, format, PushSrc::kRow, 0, 0, n, fs}) : HBD_ERR_ARG; }

int hbd_set_nco(hbd_decoder* h, int ch, double freq_hz)
{
    if (!h || ch < -1 || ch >= h->n_ch) return HBD_ERR_ARG;
    std::lock_guard<std::mutex> l(h->mtx);
    for (int c = (ch < 0 ? 0 : ch); c < (ch < 0 ? h->n_ch : ch + 1); ++c) h->hc[size_t(c)].nco_freq = freq_hz;
    if (freq_hz != 0) h->nco_any = true;
    return HBD_OK;
}
double hbd_get_nco(hbd_decoder* h, int ch)
{
    if (!h || ch < 0 || ch >= h->n_ch) return 0;
    std::lock_guard<std::mutex> l(h->mtx);
    return h->hc[size_t(ch)].nco_freq;
}

int hbd_process_async(hbd_decoder* h) { HBD_CHECK_H(h); return locked_then_fire(h, [h] { return h->process_async_locked(); }); }
int hbd_collect(hbd_decoder* h) { HBD_CHECK_H(h); return locked_then_fire(h, [h] { return h->collect_locked(0); }); }
int hbd_collect_ready(hbd_decoder* h, unsigned lag) { HBD_CHECK_H(h); return locked_then_fire(h, [h, lag] { return h->collect_locked(lag); }); }
int hbd_process(hbd_decoder* h)
{
    HBD_CHECK_H(h);
    return locked_then_fire(h, [h] {
        const int rc = h->process_async_locked();
        if (rc) return rc;
        return h->collect_locked(0);
    });
}
int hbd_reset_channels(hbd_decoder* h, const int* channels, size_t n)
{
    if (!h || (n && !channels)) return HBD_ERR_ARG;
    return locked_then_fire(h, [h, channels, n] { return h->reset_channels(channels, n); });
}
int hbd_synchronize(hbd_decoder* h)
{
    HBD_CHECK_H(h);
    std::lock_guard<std::mutex> l(h->mtx);
    return h->settle();
}
unsigned long long hbd_kernel_launches(hbd_decoder* h) { return h ? h->launches : 0; }

int hbd_set_kernel_timing(hbd_decoder* h, int on)
{
    HBD_CHECK_H(h);
    std::lock_guard<std::mutex> l(h->mtx);
    h->timing = on < 0 ? 0 : on;
    h->ev_used_k1 = h->ev_used_rest = 0;
    h->drain_host_ms = 0; h->drain_calls = 0;
    h->plan_host_ms = 0; h->plan_steps = 0;
    if (on) {   // events are created here, not on the issue path of the calls being measured
        cudaSetDevice(h->device);
        for (auto* pool : {&h->ev_k1, &h->ev_rest})
            while (pool->size() < 1024) { Event e; if (event_create(e, cudaEventDefault) != cudaSuccess) return HBD_ERR_CUDA; pool->push_back(std::move(e)); }
    }
    return HBD_OK;
}

int hbd_get_kernel_timing(hbd_decoder* h, int which, double* total_ms, unsigned* count)
{
    HBD_CHECK_H(h);
    std::lock_guard<std::mutex> l(h->mtx);
    if (h->settle()) return HBD_ERR_CUDA;
    double tot = 0; unsigned cnt = 0;
    if (which == 5) {   // host time spent replaying drained calls through the sentence layer (wall clock of the caller's thread)
        if (total_ms) *total_ms = h->drain_host_ms;
        if (count) *count = h->drain_calls;
        return HBD_OK;
    }
    if (which == 6) {   // host time of the calls' planning (plan_call), and the frame counters it stepped
        if (total_ms) *total_ms = h->plan_host_ms;
        if (count) *count = h->plan_steps;
        return HBD_OK;
    }
    if (which >= 2) {   // pipeline diagnostics (one channel group): signed gaps between events of different pairs
        const size_t calls = std::min(h->ev_used_k1, h->ev_used_rest) / 2;
        for (size_t i = 0; i < calls; ++i) {
            cudaEvent_t a = nullptr, b = nullptr;
            if (which == 2 && i + 1 < calls) { a = h->ev_k1[2 * i + 1].get(); b = h->ev_k1[2 * i + 2].get(); }        // K1 end -> next K1 start
            else if (which == 3) { a = h->ev_k1[2 * i + 1].get(); b = h->ev_rest[2 * i].get(); }                      // K1 end -> own tail start
            else if (which == 4 && i + 2 < calls) { a = h->ev_rest[2 * i + 1].get(); b = h->ev_k1[2 * i + 4].get(); } // tail end -> K1 start two calls on
            if (!a) continue;
            float ms = 0;
            if (cudaEventElapsedTime(&ms, a, b) != cudaSuccess) return HBD_ERR_CUDA;
            tot += ms; ++cnt;
        }
        if (total_ms) *total_ms = tot;
        if (count) *count = cnt;
        return HBD_OK;
    }
    const std::vector<Event>& pool = which == 0 ? h->ev_k1 : h->ev_rest;
    const size_t used = which == 0 ? h->ev_used_k1 : h->ev_used_rest;
    for (size_t i = 0; i + 1 < used; i += 2) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, pool[i].get(), pool[i + 1].get()) != cudaSuccess) return HBD_ERR_CUDA;
        tot += ms; ++cnt;
    }
    if (total_ms) *total_ms = tot;
    if (count) *count = cnt;
    return HBD_OK;
}

static size_t copy_out(const std::string& s, char* out, size_t cap)
{
    if (out && cap) memcpy(out, s.data(), std::min(cap, s.size()));
    return s.size();
}

size_t hbd_get_rtty(hbd_decoder* h, int ch, char* out, size_t cap)
{
    if (!h || ch < 0 || ch >= h->n_ch) return 0;
    std::lock_guard<std::mutex> l(h->mtx);
    return copy_out(h->text[size_t(ch)].text_stream, out, cap);
}
size_t hbd_get_last_sentence(hbd_decoder* h, int ch, char* out, size_t cap)
{
    if (!h || ch < 0 || ch >= h->n_ch) return 0;
    std::lock_guard<std::mutex> l(h->mtx);
    return copy_out(h->text[size_t(ch)].last_sentence, out, cap);
}
size_t hbd_poll_chars(hbd_decoder* h, int ch, char* out, size_t cap)
{
    if (!h || ch < 0 || ch >= h->n_ch) return 0;
    std::lock_guard<std::mutex> l(h->mtx);
    TextChannel& tc = h->text[size_t(ch)];
    hbd_result_record& pr = h->pend[size_t(ch)];
    const size_t n = tc.chars_size(pr);
    if (out && cap && n) { const std::string s = tc.chars_from(pr, 0); memcpy(out, s.data(), std::min(cap, n)); }
    if (out && cap >= n) tc.clear_chars(pr);
    return n;
}
size_t hbd_poll_sentences(hbd_decoder* h, int ch, char* out, size_t cap)
{
    if (!h || ch < 0 || ch >= h->n_ch) return 0;
    std::lock_guard<std::mutex> l(h->mtx);
    TextChannel& tc = h->text[size_t(ch)];
    hbd_result_record& pr = h->pend[size_t(ch)];
    const size_t n = tc.sent_size(pr);
    if (out && cap && n) { const std::string s = tc.sentences_all(pr); memcpy(out, s.data(), std::min(cap, n)); }
    if (out && cap >= n) tc.clear_sentences(pr);
    return n;
}
size_t hbd_poll_raw_chars(hbd_decoder* h, int ch, unsigned char* out, size_t cap)
{
    if (!h || ch < 0 || ch >= h->n_ch) return 0;
    std::lock_guard<std::mutex> l(h->mtx);
    auto& v = h->text[size_t(ch)].raw_pending;
    const size_t n = v.size();
    if (out && cap) memcpy(out, v.data(), std::min(cap, n));
    if (out && cap >= n) v.clear();
    return n;
}
int hbd_set_host_threads(hbd_decoder* h, int n)
{
    HBD_CHECK_H(h); std::lock_guard<std::mutex> l(h->mtx); h->host_threads = std::max(1, std::min(n, 64)); return HBD_OK;
}
int hbd_set_raw_chars(hbd_decoder* h, int on)
{
    HBD_CHECK_H(h); std::lock_guard<std::mutex> l(h->mtx); h->keep_raw = on != 0; return HBD_OK;
}
int hbd_attach_tracker(hbd_decoder* h, hbd_tracker* t, int ch_offset)
{
    HBD_CHECK_H(h); std::lock_guard<std::mutex> l(h->mtx); h->tracker = t; h->tracker_off = ch_offset; return HBD_OK;
}

int hbd_set_sentence_callback(hbd_decoder* h, hbd_sentence_cb cb, void* user)
{
    HBD_CHECK_H(h); std::lock_guard<std::mutex> l(h->mtx); h->sentence_cb = cb; h->sentence_user = user; return HBD_OK;
}
int hbd_set_chars_callback(hbd_decoder* h, hbd_chars_cb cb, void* user)
{
    HBD_CHECK_H(h); std::lock_guard<std::mutex> l(h->mtx); h->chars_cb = cb; h->chars_user = user; return HBD_OK;
}

// ---- SSDV packet sync ---------------------------------------------------------------------------------------
int hbd_set_ssdv(hbd_decoder* h, int on)
{
    HBD_CHECK_H(h);
    return locked_then_fire(h, [h, on] { return h->enable_ssdv(on != 0); });
}
int hbd_set_ssdv_callback(hbd_decoder* h, hbd_ssdv_cb cb, void* user)
{
    HBD_CHECK_H(h);
    return locked_then_fire(h, [h, cb, user] {
        const int rc = cb ? h->enable_ssdv(true) : HBD_OK;   // drains the calls in flight (under the previous callback)
        h->ssdv_cb = cb; h->ssdv_user = user;
        return rc;
    });
}
size_t hbd_poll_ssdv_packets(hbd_decoder* h, int ch, hbd_ssdv_packet_info* infos, unsigned char* packets, size_t cap_packets)
{
    if (!h || ch < 0 || ch >= h->n_ch) return 0;
    std::lock_guard<std::mutex> l(h->mtx);
    if (h->ssdv.empty()) return 0;
    auto& ev = h->ssdv[size_t(ch)].events_pending;
    const size_t n = ev.size();
    for (size_t i = 0; i < std::min(n, cap_packets); ++i) {
        if (infos) fill_ssdv_info(infos[i], ev[i]);
        if (packets) memcpy(packets + 256 * i, ev[i].data.data(), 256);
    }
    if ((infos || packets) && cap_packets >= n) ev.clear();
    return n;
}
size_t hbd_get_ssdv_image(hbd_decoder* h, int ch, const char* callsign, int image_id, unsigned char* out, size_t cap)
{
    if (!h || ch < 0 || ch >= h->n_ch || !callsign) return 0;
    std::lock_guard<std::mutex> l(h->mtx);
    if (h->ssdv.empty()) return 0;
    return h->ssdv[size_t(ch)].image(callsign, image_id, out, cap);
}
int hbd_get_ssdv_last_image(hbd_decoder* h, int ch, char callsign[8], int* image_id)
{
    HBD_CHECK_CH(h, ch); std::lock_guard<std::mutex> l(h->mtx);
    if (h->ssdv.empty()) return HBD_ERR_STATE;
    const auto& k = h->ssdv[size_t(ch)].last_key;
    if (callsign) { memset(callsign, 0, 8); strncpy(callsign, k.first.c_str(), 7); }
    if (image_id) *image_id = k.second;
    return HBD_OK;
}
int hbd_ssdv_check_packets(hbd_decoder* h, unsigned char* windows, size_t n, int* verdict, int* errors)
{
    HBD_CHECK_H(h);
    if (!windows || !verdict || !errors) return HBD_ERR_ARG;
    if (!n) return HBD_OK;
    std::lock_guard<std::mutex> l(h->mtx);
    if (cudaSetDevice(h->device) != cudaSuccess) return HBD_ERR_CUDA;
    DevPtr<unsigned char> w; DevPtr<int> v;
    auto fail = [&](const char* what) { h->set_error(what); return HBD_ERR_CUDA; };
    if (dev_alloc(w, n * 256) != cudaSuccess || dev_alloc(v, n * 2) != cudaSuccess) return fail("cudaMalloc (ssdv check)");
    unsigned char* d_w = w.get(); int* d_v = v.get();
    if (cudaMemcpyAsync(d_w, windows, n * 256, cudaMemcpyHostToDevice, h->stream) != cudaSuccess) return fail("cudaMemcpyAsync (ssdv check)");
    int nl = 0;
    if (launch_ssdv_check(d_w, int(n), d_v, d_v + n, h->stream, &nl) != cudaSuccess) return fail("ssdv_check_kernel launch");
    h->launches += unsigned(nl);
    if (cudaMemcpyAsync(windows, d_w, n * 256, cudaMemcpyDeviceToHost, h->stream) != cudaSuccess ||
        cudaMemcpyAsync(verdict, d_v, n * sizeof(int), cudaMemcpyDeviceToHost, h->stream) != cudaSuccess ||
        cudaMemcpyAsync(errors, d_v + n, n * sizeof(int), cudaMemcpyDeviceToHost, h->stream) != cudaSuccess ||
        cudaStreamSynchronize(h->stream) != cudaSuccess) return fail("ssdv check read-back");
    return HBD_OK;
}

// host half of the SSDV path alone (test hook, no GPU): replay SsdvChannel over `n_chunks` pushes of the character
// stream `chars`, with the accepted windows given by position
size_t hbd_ssdv_host_replay(const unsigned char* chars, const size_t* chunk_sizes, size_t n_chunks, const unsigned* accepted_pos,
                            const unsigned char* accepted_packets, const int* accepted_errors, size_t n_accepted,
                            hbd_ssdv_packet_info* out_infos, unsigned* out_chunk, unsigned char* out_packets, size_t cap)
{
    if (!chars || !chunk_sizes) return 0;
    SsdvChannel sc;
    for (size_t i = 0; i < n_accepted; ++i) {
        SsdvVerdict v; v.pos = accepted_pos[i]; v.errors = accepted_errors ? accepted_errors[i] : 0;
        memcpy(v.data.data(), accepted_packets + 256 * i, 256);
        sc.verdicts.push_back(v);
    }
    size_t off = 0, n_ev = 0;
    for (size_t c = 0; c < n_chunks; ++c) {
        SsdvEvent ev;
        if (chunk_sizes[c] && sc.push(chars + off, chunk_sizes[c], ev)) {
            if (n_ev < cap) {
                if (out_infos) fill_ssdv_info(out_infos[n_ev], ev);
                if (out_chunk) out_chunk[n_ev] = unsigned(c);
                if (out_packets) memcpy(out_packets + 256 * n_ev, ev.data.data(), 256);
            }
            ++n_ev;
        }
        off += chunk_sizes[c];
    }
    return n_ev;
}

int hbd_get_decimation_factor(hbd_decoder* h) { if (!h) return 0; std::lock_guard<std::mutex> l(h->mtx); return h->factor; }
double hbd_get_input_sampling_rate(hbd_decoder* h) { if (!h) return 0; std::lock_guard<std::mutex> l(h->mtx); return h->fs_in; }
double hbd_get_decimated_sampling_rate(hbd_decoder* h) { if (!h) return 0; std::lock_guard<std::mutex> l(h->mtx); return h->fs_in / h->factor; }
double hbd_get_symbol_rate(hbd_decoder* h, int ch) { return hbd_get_baud(h, ch); }
int hbd_n_channels(hbd_decoder* h) { return h ? h->n_ch : 0; }
size_t hbd_get_bins_count(hbd_decoder* h) { if (!h) return size_t(kFftN); std::lock_guard<std::mutex> l(h->mtx); return size_t(h->fft_n); }

// min(n, cap) floats from the device into out (the caller has settled the handle); returns n, or 0 when the copy fails
static size_t fetch_floats(const void* dsrc, size_t n, float* out, size_t cap)
{
    if (out && cap && n && cudaMemcpy(out, dsrc, std::min(n, cap) * sizeof(float), cudaMemcpyDeviceToHost) != cudaSuccess) return 0;
    return n;
}

size_t hbd_get_fft(hbd_decoder* h, int ch, float* out, size_t cap)
{
    if (!h || ch < 0 || ch >= h->n_ch) return 0;
    std::lock_guard<std::mutex> l(h->mtx);
    ChanState st;
    if (h->read_states(size_t(ch), 1, &st) || !st.have_spectrum) return 0; // freq_out_ is empty before the first FFT
    return fetch_floats(h->fft.spectrum.get() + size_t(ch) * size_t(h->fft_n), 2 * size_t(h->fft_n), out, cap);
}
size_t hbd_get_power_spectrum(hbd_decoder* h, int ch, float* out, size_t cap)
{
    if (!h || ch < 0 || ch >= h->n_ch) return 0;
    std::lock_guard<std::mutex> l(h->mtx);
    ChanState st;
    if (h->read_states(size_t(ch), 1, &st) || !st.have_spectrum) return 0;
    return fetch_floats(h->fft.power.get() + size_t(ch) * size_t(h->fft_n), size_t(h->fft_n), out, cap);
}
size_t hbd_get_demodulated(hbd_decoder* h, int ch, float* out, size_t cap)
{
    if (!h || ch < 0 || ch >= h->n_ch) return 0;
    std::lock_guard<std::mutex> l(h->mtx);
    h->sync_ctrs();
    const size_t n = h->hc[size_t(ch)].demod_n;   // a call that demodulates nothing leaves the previous block in place
    if (!h->demod.get() || h->settle()) return 0;
    return fetch_floats(h->demod.get() + size_t(ch) * h->demod.pitch, n, out, cap);
}
int hbd_get_peaks(hbd_decoder* h, int ch, int* pl, int* pr)
{
    HBD_CHECK_CH(h, ch); std::lock_guard<std::mutex> l(h->mtx);
    ChanState st; const int rc = h->read_states(size_t(ch), 1, &st); if (rc) return rc;
    if (pl) *pl = st.gui_left; if (pr) *pr = st.gui_right; return HBD_OK;
}
int hbd_get_noise_floor(hbd_decoder* h, int ch, double* nf, double* nv)
{
    HBD_CHECK_CH(h, ch); std::lock_guard<std::mutex> l(h->mtx);
    ChanState st; const int rc = h->read_states(size_t(ch), 1, &st); if (rc) return rc;
    if (nf) *nf = st.afc_noise_floor; if (nv) *nv = st.afc_noise_var; return HBD_OK;
}
double hbd_get_shift(hbd_decoder* h, int ch)
{
    if (!h || ch < 0 || ch >= h->n_ch) return 0; std::lock_guard<std::mutex> l(h->mtx);
    ChanState st; if (h->read_states(size_t(ch), 1, &st)) return 0; return st.afc_shift_hz;
}
double hbd_get_frequency_correction(hbd_decoder* h, int ch)
{
    if (!h || ch < 0 || ch >= h->n_ch) return 0; std::lock_guard<std::mutex> l(h->mtx);
    ChanState st; if (h->read_states(size_t(ch), 1, &st)) return 0; return st.afc_correction;
}
int hbd_reset_frequency_correction(hbd_decoder* h, int ch, double corr)
{
    HBD_CHECK_CH(h, ch); std::lock_guard<std::mutex> l(h->mtx);
    cudaSetDevice(h->device);
    // ordered after everything in flight, like a call between two process() calls
    if (h->sync_groups() || launch_afc_reset(h->d_state.get(), ch, corr, h->fs_in / h->factor, h->fft_n, h->stream) != cudaSuccess) return HBD_ERR_CUDA;
    ++h->launches;
    return cudaStreamSynchronize(h->stream) == cudaSuccess ? HBD_OK : HBD_ERR_CUDA;
}
// ---- websocket wire formats ---------------------------------------------------------------------------------
int hbd_decoder::ensure_frames(size_t pitch)
{
    if (pitch <= frames_pitch && d_frames) return HBD_OK;
    pitch = (pitch + 255) & ~size_t(255);
    DevPtr<unsigned char> frames;
    HBD_CUDA_CHECK(dev_alloc(frames, size_t(n_ch) * pitch));
    d_frames = std::move(frames); frames_pitch = pitch;
    return HBD_OK;
}

// accumulation buffers: 50 symbols of the slowest channel plus one call's worth of new samples
int hbd_decoder::ensure_dacc()
{
    const double fs_dec = fs_in / factor;
    size_t need = 0;
    for (const auto& x : hc) if (x.baud > 0) need = std::max(need, size_t(fs_dec / x.baud * 50));
    need += demod.pitch + 64;
    if (need > dacc.pitch) {
        if (sync_groups()) return HBD_ERR_CUDA;
        HBD_CUDA_CHECK(dacc.grow((need + 15) & ~size_t(15), size_t(n_ch), dacc.pitch, stream));
    }
    return HBD_OK;
}

extern "C" int hbd_set_demod_accumulate(hbd_decoder* h, int on)
{
    HBD_CHECK_H(h);
    std::lock_guard<std::mutex> l(h->mtx);
    h->demod_acc_on = on != 0;
    return HBD_OK;
}

// frames of channels [ch0, ch0 + nc) into the device scratch, then one copy of sizes + one of payloads
static size_t fetch_frames(hbd_decoder* h, int ch0, int nc, bool spectrum, float zoom, int resolution, int type_size,
                           unsigned char* out, size_t pitch, unsigned* sizes)
{
    if (type_size != 1 && type_size != 2 && type_size != 4) return 0;
    if (resolution < 0) resolution = 0;
    if (h->settle()) return 0;
    const size_t hdr = spectrum ? size_t(kSpectrumHeaderBytes) : size_t(kDemodHeaderBytes);
    const size_t max_n = spectrum ? size_t(h->fft_n) : std::max<size_t>(h->dacc.pitch, 1);
    const size_t need = hdr + std::min<size_t>(max_n, size_t(resolution)) * size_t(type_size);
    if (h->ensure_frames(need)) return 0;
    int nl = 0;
    cudaError_t e;
    if (spectrum) {
        SpectrumFrameArgs a{};
        a.state = h->d_state.get(); a.power = h->fft.power.get(); a.fft_n = h->fft_n; a.fs_dec = h->fs_in / h->factor; a.zoom = zoom; a.resolution = resolution; a.type_size = type_size;
        a.out = h->d_frames.get(); a.out_pitch = h->frames_pitch; a.sizes = h->d_frame_sizes.get(); a.ch0 = ch0;
        e = launch_spectrum_frames(a, nc, h->stream, &nl);
    } else {
        if (!h->dacc.get()) return 0;
        DemodFrameArgs a{};
        a.acc = h->dacc.get(); a.acc_pitch = h->dacc.pitch; a.acc_n = h->d_dacc_n.get(); a.resolution = resolution; a.type_size = type_size;
        a.out = h->d_frames.get(); a.out_pitch = h->frames_pitch; a.sizes = h->d_frame_sizes.get(); a.ch0 = ch0;
        e = launch_demod_frames(a, nc, h->stream, &nl);
    }
    h->launches += unsigned(nl);
    if (e != cudaSuccess) { h->set_error(cudaGetErrorString(e)); return 0; }
    if (cudaMemcpyAsync(h->h_frame_sizes.data(), h->d_frame_sizes.get(), sizeof(unsigned) * size_t(nc), cudaMemcpyDeviceToHost, h->stream) != cudaSuccess) return 0;
    if (cudaStreamSynchronize(h->stream) != cudaSuccess) return 0;
    size_t longest = 0;
    for (int i = 0; i < nc; ++i) longest = std::max<size_t>(longest, h->h_frame_sizes[size_t(i)]);
    if (sizes) for (int i = 0; i < nc; ++i) sizes[i] = h->h_frame_sizes[size_t(i)];
    if (out && pitch && longest) {
        const size_t w = std::min(pitch, longest);
        if (cudaMemcpy2D(out, pitch, h->d_frames.get(), h->frames_pitch, w, size_t(nc), cudaMemcpyDeviceToHost) != cudaSuccess) return 0;
    }
    return longest;
}

extern "C" {
size_t hbd_get_spectrum_frame(hbd_decoder* h, int ch, float zoom, int resolution, int type_size, unsigned char* out, size_t cap)
{
    if (!h || ch < 0 || ch >= h->n_ch) return 0;
    std::lock_guard<std::mutex> l(h->mtx);
    return fetch_frames(h, ch, 1, true, zoom, resolution, type_size, out, cap, nullptr);
}
size_t hbd_get_spectrum_frames(hbd_decoder* h, float zoom, int resolution, int type_size, unsigned char* out, size_t pitch, unsigned* sizes)
{
    if (!h) return 0;
    std::lock_guard<std::mutex> l(h->mtx);
    return fetch_frames(h, 0, h->n_ch, true, zoom, resolution, type_size, out, pitch, sizes);
}
size_t hbd_get_demod_frame(hbd_decoder* h, int ch, int resolution, int type_size, unsigned char* out, size_t cap)
{
    if (!h || ch < 0 || ch >= h->n_ch) return 0;
    std::lock_guard<std::mutex> l(h->mtx);
    return fetch_frames(h, ch, 1, false, 0.f, resolution, type_size, out, cap, nullptr);
}
size_t hbd_get_demod_frames(hbd_decoder* h, int resolution, int type_size, unsigned char* out, size_t pitch, unsigned* sizes)
{
    if (!h) return 0;
    std::lock_guard<std::mutex> l(h->mtx);
    return fetch_frames(h, 0, h->n_ch, false, 0.f, resolution, type_size, out, pitch, sizes);
}
} // extern "C"

// AFC loop closed on the GPU for all channels (see afc_retune_kernel); returns the number of channels retuned
int hbd_afc_retune(hbd_decoder* h, double min_abs_hz, double* applied_out)
{
    HBD_CHECK_H(h);
    std::lock_guard<std::mutex> l(h->mtx);
    cudaSetDevice(h->device);
    if (h->sync_groups()) return HBD_ERR_CUDA;
    const size_t n = size_t(h->n_ch);
    DevPtr<double> d_applied;
    std::vector<double> applied(n, 0.0);
    cudaError_t e = dev_alloc(d_applied, n);
    if (e == cudaSuccess) {
        e = launch_afc_retune(h->d_state.get(), h->n_ch, min_abs_hz, h->fs_in / h->factor, d_applied.get(), h->fft_n, h->stream);
        ++h->launches;
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(applied.data(), d_applied.get(), n * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) { h->set_error(cudaGetErrorString(e)); return HBD_ERR_CUDA; }
    int count = 0;
    for (size_t c = 0; c < n; ++c) {
        if (applied[c] != 0.0) { h->hc[c].nco_freq += applied[c]; h->nco_any = true; ++count; }
        if (applied_out) applied_out[c] = applied[c];
    }
    return count;
}
int hbd_set_baud_estimation(hbd_decoder* h, int on)
{
    HBD_CHECK_H(h);
    std::lock_guard<std::mutex> l(h->mtx);
    if ((on != 0) == h->baud_on) return HBD_OK;
    if (cudaSetDevice(h->device) != cudaSuccess) return HBD_ERR_CUDA;
    if (on) {
        h->baud_on = true; h->baud_fs = 0;
        const int rc = h->fs_in ? h->baud_start() : HBD_OK;   // otherwise at the first call
        if (rc) h->baud_on = false;
        return rc;
    }
    if (h->sync_groups()) { h->set_error("stream sync failed"); return HBD_ERR_CUDA; }
    h->baud_on = false; h->baud_fs = 0; h->baud_lmax = 0;
    h->d_bhist.reset(); h->d_btrack.reset(); h->d_best.reset();
    return HBD_OK;
}
int hbd_get_baud_estimates(hbd_decoder* h, hbd_baud_estimate* out, size_t cap)
{
    HBD_CHECK_H(h);
    std::lock_guard<std::mutex> l(h->mtx);
    if (!h->baud_on) { h->set_error("baud estimation is off"); return HBD_ERR_STATE; }
    std::vector<hbd_baud_estimate> est;
    if (out && cap) {
        const int rc = h->baud_estimates(est);
        if (rc) return rc;
        memcpy(out, est.data(), std::min(cap, est.size()) * sizeof(hbd_baud_estimate));
    }
    return h->n_ch;
}
int hbd_apply_baud_estimates(hbd_decoder* h, double min_confidence, unsigned min_runs, double* applied)
{
    HBD_CHECK_H(h);
    std::lock_guard<std::mutex> l(h->mtx);
    if (!h->baud_on) { h->set_error("baud estimation is off"); return HBD_ERR_STATE; }
    std::vector<hbd_baud_estimate> est;
    { const int rc = h->baud_estimates(est); if (rc) return rc; }
    int count = 0;
    for (size_t c = 0; c < est.size(); ++c) {
        const hbd_baud_estimate& e = est[c];
        const bool set = e.nominal > 0 && e.runs >= min_runs && e.confidence >= min_confidence && e.nominal != h->hc[c].baud;
        if (set) { h->hc[c].baud = e.nominal; h->hc[c].cfg_dirty = true; ++count; }   // what hbd_set_baud(h, c, nominal) does
        if (applied) applied[c] = set ? e.nominal : 0.0;
    }
    if (count) h->cfg_dirty_any = h->derived_dirty = true;
    return count;
}
size_t hbd_get_baud_histogram(hbd_decoder* h, int ch, unsigned* out, size_t cap)
{
    if (!h || ch < 0 || ch >= h->n_ch) return 0;
    std::lock_guard<std::mutex> l(h->mtx);
    if (!h->baud_on || !h->fs_in || cudaSetDevice(h->device) != cudaSuccess || h->baud_start() || h->settle()) return 0;
    const size_t len = size_t(h->baud_lmax) + 1;
    if (out && cap && cudaMemcpy(out, h->d_bhist.get() + size_t(ch) * len, std::min(cap, len) * sizeof(unsigned), cudaMemcpyDeviceToHost) != cudaSuccess) return 0;
    return len;
}

// all channels in one device->host copy: out[ch*6 + {0..5}] = correction, shift, noise floor, noise variance, peak l, peak r
size_t hbd_get_stats_batch(hbd_decoder* h, double* out, size_t cap_doubles)
{
    if (!h) return 0;
    std::lock_guard<std::mutex> l(h->mtx);
    const size_t n = size_t(h->n_ch);
    if (!out || cap_doubles < 6 * n) return 6 * n;
    std::vector<ChanState> st(n);
    if (h->read_states(0, n, st.data())) return 0;
    for (size_t c = 0; c < n; ++c) afc_scalars(st[c], out + 6 * c);
    return 6 * n;
}

// one query under one lock: the spectrum and the scalars come from the same completed call
size_t hbd_get_spectrum_info(hbd_decoder* h, int ch, hbd_spectrum_info* info, float* power, size_t cap)
{
    if (!h || ch < 0 || ch >= h->n_ch || !info) return 0;
    memset(info, 0, sizeof(*info));
    std::lock_guard<std::mutex> l(h->mtx);
    ChanState st;
    if (h->read_states(size_t(ch), 1, &st) || !st.have_spectrum) return 0; // Decoder.h:818-819
    std::vector<float> p(size_t(h->fft_n));
    if (!fetch_floats(h->fft.power.get() + size_t(ch) * p.size(), p.size(), p.data(), p.size())) return 0;
    info->min_ = *std::min_element(p.begin(), p.end());
    info->max_ = *std::max_element(p.begin(), p.end());
    info->peak_left_ = std::abs(st.gui_left); info->peak_left_valid_ = st.gui_left > 0;
    info->peak_right_ = std::abs(st.gui_right); info->peak_right_valid_ = st.gui_right > 0;
    info->noise_floor_ = st.afc_noise_floor; info->noise_variance_ = st.afc_noise_var;
    info->sampling_rate_ = h->fs_in / h->factor;
    info->shift_ = st.afc_shift_hz;
    if (power && cap) memcpy(power, p.data(), std::min(cap, p.size()) * sizeof(float));
    return p.size();
}

size_t hbd_debug_stage(hbd_decoder* h, int ch, int stage, float* out, size_t cap)
{
    if (!h || ch < 0 || ch >= h->n_ch) return 0;
    std::lock_guard<std::mutex> l(h->mtx);
    h->sync_ctrs();
    const HostChan& x = h->hc[size_t(ch)];
    switch (stage) {
    case HBD_STAGE_DECIMATED:
        if (!h->rec.get(0) || h->settle()) return 0;
        return fetch_floats(h->rec.get(0) + size_t(ch) * h->rec.pitch, 2 * size_t(x.last_n2), out, cap);
    case HBD_STAGE_FILTERED:
        if (!h->rec.get(1) || h->settle()) return 0;
        return fetch_floats(h->rec.get(1) + size_t(ch) * h->rec.pitch, 2 * size_t(x.last_nf), out, cap);
    case HBD_STAGE_DEMOD:
        if (!h->demod.get() || h->settle()) return 0;
        return fetch_floats(h->demod.get() + size_t(ch) * h->demod.pitch, size_t(x.last_nf), out, cap);
    case HBD_STAGE_LPTAPS:
        if (h->settle()) return 0;
        return fetch_floats(h->d_lptaps.get() + size_t(ch) * kLpMaxTaps, x.lp_ntaps, out, cap);
    case HBD_STAGE_PENDING: {
        ChanState st;
        if (!h->slicer.get() || h->read_states(size_t(ch), 1, &st)) return 0;
        return fetch_floats(h->slicer.get() + size_t(ch) * h->slicer.pitch, st.slicer_n, out, cap);
    }
    case HBD_STAGE_BITS: {
        if (!h->d_rec_bits.get() || h->settle()) return 0;
        unsigned nb = 0;
        if (cudaMemcpy(&nb, h->d_rec_bits_n.get() + ch, 4, cudaMemcpyDeviceToHost) != cudaSuccess) return 0;
        nb = std::min(nb, h->rec_bits_pitch);
        if (out && cap && nb) {
            std::vector<unsigned char> b(nb);
            if (cudaMemcpy(b.data(), h->d_rec_bits.get() + size_t(ch) * h->rec_bits_pitch, nb, cudaMemcpyDeviceToHost) != cudaSuccess) return 0;
            for (size_t i = 0; i < std::min<size_t>(nb, cap); ++i) out[i] = float(b[i]);
        }
        return nb;
    }
    default: return 0;
    }
}

size_t hbd_design_lowpass(float rel_width, float trans, size_t input_size, size_t current_taps, float* out, size_t cap)
{
    std::vector<float> taps;
    const size_t T = design_lowpass(rel_width, trans, input_size, current_taps, taps);
    if (out && T != current_taps) memcpy(out, taps.data(), std::min(cap, taps.size()) * sizeof(float));
    return T;
}

int hbd_extract_sentence(const char* stream, size_t n, char* callsign, char* data, char* crc, size_t cap, size_t* rest)
{
    SentenceMatch m;
    if (!extract_sentence(std::string(stream, n), m)) return 0;
    auto put = [cap](char* dst, const std::string& s) { if (dst && cap) { const size_t k = std::min(cap - 1, s.size()); memcpy(dst, s.data(), k); dst[k] = 0; } };
    put(callsign, m.callsign); put(data, m.data); put(crc, m.crc);
    if (rest) *rest = m.rest_offset;
    return 1;
}

// the text layer alone (test hook, no GPU): TextChannel::feed over n_chunks pushes of raw characters; `out` receives
// "<CRC-valid sentences, one per line>\x1e<last sentence>\x1e<text stream>"; returns the size of that report
size_t hbd_text_replay(const unsigned char* chars, const size_t* chunk_sizes, size_t n_chunks, char* out, size_t cap)
{
    if (!chars || !chunk_sizes) return 0;
    TextChannel tc;
    hbd_result_record pr; memset(&pr, 0, sizeof(pr));
    size_t off = 0;
    for (size_t c = 0; c < n_chunks; ++c) { tc.feed(chars + off, chunk_sizes[c], 0, SentenceSink(), true, pr); off += chunk_sizes[c]; }
    const std::string rep = tc.sentences_all(pr) + "\x1e" + tc.last_sentence + "\x1e" + tc.text_stream;
    if (out && cap) memcpy(out, rep.data(), std::min(cap, rep.size()));
    return rep.size();
}

void hbd_crc16(const char* s, size_t n, char out[5])
{
    const std::string r = crc16_hex(std::string(s, n));
    memcpy(out, r.data(), 4); out[4] = 0;
}

} // extern "C"
