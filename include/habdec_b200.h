/* habdec_b200 -- C ABI of the B200-native batched RTTY decoder.
 *
 * One hbd_decoder = N independent channels, each behaving like one reference
 * habdec::Decoder<float> (code/Decoder/Decoder.h:51-203 under /root/reference).
 * Every entry point names the reference member it replaces.  Plain C types only;
 * the library is libhabdec_b200.so (CUDA, sm_100a).  There is no CPU fallback:
 * every call fails with HBD_ERR_CUDA when no usable device is present.
 *
 * Threading model follows the reference (Decoder.h:146-196): one thread feeds
 * and processes, other threads may call getters/setters; all entry points take
 * the handle's mutex.  Callbacks fire on the thread that called hbd_process() /
 * hbd_collect*() AFTER the mutex has been released, so a callback may call any
 * hbd_* function of the same handle (like the reference's callbacks may call
 * getRTTY()/getLastSentence()).  hbd_last_error() returns a pointer that the next
 * failing call on the handle overwrites.
 *
 * Batch-wide by design: the input sampling rate and the decimation plan are
 * shared by all channels of a handle (they are channels of one capture / one
 * receiver type); everything else is per channel.  `ch == -1` in a setter
 * means "all channels".
 */
#ifndef HABDEC_B200_H
#define HABDEC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct hbd_decoder hbd_decoder;

enum {
    HBD_OK          = 0,
    HBD_ERR_ARG     = -1,  /* bad channel index / pointer / size */
    HBD_ERR_CUDA    = -2,  /* CUDA runtime error, see hbd_last_error() */
    HBD_ERR_STATE   = -3,  /* call not valid in the current state */
    HBD_ERR_NOMEM   = -4
};

/* SpectrumInfo<float> scalars, code/Decoder/SpectrumInfo.h:35-85 + Decoder.h:814-836 */
typedef struct hbd_spectrum_info {
    float  min_, max_;
    double noise_floor_, noise_variance_, sampling_rate_, shift_;
    int    peak_left_, peak_right_;
    int    peak_left_valid_, peak_right_valid_;
} hbd_spectrum_info;

/* callbacks fire on the thread that calls hbd_process(), like the reference's
 * sentence_callback_ / character_callback_ (Decoder.h:135,138,604-606,625-626) */
typedef void (*hbd_sentence_cb)(void* user, int ch, const char* callsign, const char* data, const char* crc);
typedef void (*hbd_chars_cb)(void* user, int ch, const char* chars, size_t n);

/* ---- life cycle ------------------------------------------------------------------------------------- */
int  hbd_create(int n_channels, int cuda_device, hbd_decoder** out);
void hbd_destroy(hbd_decoder* h);
const char* hbd_last_error(hbd_decoder* h);
/* run all work on this cudaStream_t (default: a private non-blocking stream) */
int  hbd_set_stream(hbd_decoder* h, void* cuda_stream);
/* spectrum / AFC FFT size: 4096 (the reference's fft_bins_cnt_, Decoder.h:163; default) or 16384 (the 16k-bin
 * spectrum of BASELINE configs[1]).  Restarts spectrum collection and the AFC averages of every channel.
 * On failure the previous size, spectra and AFC averages stay in force. */
int  hbd_set_fft_size(hbd_decoder* h, size_t n_bins);
/* keep per-call stage arrays (decimated IQ, filtered IQ, slicer bits) for hbd_debug_stage(); test use */
int  hbd_set_record(hbd_decoder* h, int on);

/* ---- configuration (Decoder.h:77-91) ---------------------------------------------------------------- */
int    hbd_set_baud(hbd_decoder* h, int ch, double baud);              /* Decoder::baud(double)          :656 */
double hbd_get_baud(hbd_decoder* h, int ch);                           /* Decoder::baud()                :664 */
int    hbd_set_rtty_bits(hbd_decoder* h, int ch, size_t bits);         /* Decoder::rtty_bits(size_t)     :671 */
size_t hbd_get_rtty_bits(hbd_decoder* h, int ch);
int    hbd_set_rtty_stops(hbd_decoder* h, int ch, float stops);        /* Decoder::rtty_stops(float)     :686 */
float  hbd_get_rtty_stops(hbd_decoder* h, int ch);
int    hbd_set_lowpass_bw(hbd_decoder* h, int ch, float bw_hz);        /* Decoder::lowpass_bw(float)     :238 */
float  hbd_get_lowpass_bw(hbd_decoder* h, int ch);
int    hbd_set_lowpass_trans(hbd_decoder* h, int ch, float trans);     /* Decoder::lowpass_trans(float)  :252 */
float  hbd_get_lowpass_trans(hbd_decoder* h, int ch);
int    hbd_set_dc_remove(hbd_decoder* h, int ch, int on);              /* Decoder::dc_remove(bool)       :701 */
int    hbd_get_dc_remove(hbd_decoder* h, int ch);
/* returns the new factor; the current one if out of [1,256]; 0 if not a supported power of two (:268-332) */
size_t hbd_setup_decimation_factor(hbd_decoder* h, size_t factor);
/* Decoder::setupDecimationStagesBW (:336-412); returns 0 before the first push latched a sampling rate */
/* Either setup returns 0 when the new plan cannot be installed (e.g. out of device memory): the previous plan stays in force. */
size_t hbd_setup_decimation_bw(hbd_decoder* h, double max_sampling_rate);

/* ---- feed (Decoder::pushSamples, Decoder.h:206-219).  iq = interleaved cf32, n in complex samples.
 * The first push latches the sampling rate (as float, like Decoder::init :223-225). ------------------------ */
int hbd_push_samples(hbd_decoder* h, int ch, const float* iq, size_t n_complex, double sampling_rate);
/* all channels at once: host matrix [n_channels][pitch_complex] */
int hbd_push_samples_batch(hbd_decoder* h, const float* iq, size_t n_complex, size_t pitch_complex, double sampling_rate);
/* zero copy: DEVICE matrix [n_channels][pitch_complex], 16-byte aligned rows; it must stay valid and
 * unchanged until the next hbd_process()/hbd_process_async() has completed (hbd_synchronize) */
int hbd_push_samples_device(hbd_decoder* h, const float* d_iq, size_t n_complex, size_t pitch_complex, double sampling_rate);

/* ---- integer IQ input (what receivers deliver; the reference gets cf32 from SoapySDR's CPU conversion) ---------------
 * I, Q interleaved, little endian.  The decoder sees the dequantised value, exactly representable in float32:
 *   HBD_IQ_CF32  8 B / sample   as is
 *   HBD_IQ_CS16  4 B / sample   v / 32768          (Airspy, SDRplay, SoapySDR "CS16")
 *   HBD_IQ_CS8   2 B / sample   v / 128            (HackRF)
 *   HBD_IQ_CU8   2 B / sample   (v - 128) / 128    (RTL-SDR, rtl_sdr .cu8 files)
 * so an integer push is bit for bit the cf32 push of its dequantised values.  CU8 is mapped exactly (CS8 of v ^ 0x80), not
 * re-centred: a receiver's DC offset is left to dc_remove and the NCO.  The format may change from one push to the next.
 * The five entries below mirror the cf32 ones (same rules for pending host / device pushes, queue depths and device
 * pointer lifetime); n and pitch count complex samples; HBD_IQ_CF32 makes them exactly the cf32 entry points.  Integer
 * data crosses PCIe and HBM as integers: with the /64 first stage (factor 256) and no NCO set, the decimator reads a
 * device push in place; every other path widens on the GPU into the cf32 buffers the cf32 push would have used.
 * Device matrices: 16-byte aligned, pitch * bytes a multiple of 16.  Unknown format / misalignment: HBD_ERR_ARG. */
enum hbd_iq_format { HBD_IQ_CF32 = 0, HBD_IQ_CS16 = 1, HBD_IQ_CS8 = 2, HBD_IQ_CU8 = 3 };
int hbd_push_iq(hbd_decoder* h, int ch, const void* iq, int format, size_t n_complex, double sampling_rate);
int hbd_push_iq_batch(hbd_decoder* h, const void* iq, int format, size_t n_complex, size_t pitch_complex, double sampling_rate);
int hbd_push_iq_device(hbd_decoder* h, const void* d_iq, int format, size_t n_complex, size_t pitch_complex, double sampling_rate);
int hbd_push_iq_wideband(hbd_decoder* h, const void* iq, int format, size_t n_complex, double sampling_rate);
int hbd_push_iq_wideband_device(hbd_decoder* h, const void* d_iq, int format, size_t n_complex, double sampling_rate);

/* ---- NCO pre-mixer (new; the reference retunes the SDR instead: websocketServer/main.cpp:247-265) -----------
 * Channel `ch` (-1: all) is mixed down by freq_hz before the decimator: x[i] * exp(-2 pi i f t), phase kept in
 * float64 and continuous across pushes and frequency changes.  With it, one wideband capture can feed many
 * frequency-offset channels (hbd_push_wideband*), and the AFC loop closes without touching the radio:
 *   corr = hbd_get_frequency_correction(h, ch); hbd_set_nco(h, ch, hbd_get_nco(h, ch) + corr);
 *   hbd_reset_frequency_correction(h, ch, corr);      -- same sequence as main.cpp:248-265 */
int    hbd_set_nco(hbd_decoder* h, int ch, double freq_hz);
double hbd_get_nco(hbd_decoder* h, int ch);
/* the whole loop for every channel in one call: where |frequency correction| > min_abs_hz (the reference uses
 * 100 Hz) the NCO is moved by the correction and the AFC is reset; applied[n_channels] (may be NULL) receives the
 * corrections, the return value is the number of channels retuned (< 0: error) */
int    hbd_afc_retune(hbd_decoder* h, double min_abs_hz, double* applied);
/* one capture (host / device cf32 row of n_complex samples) pushed to EVERY channel through its NCO.  With the
 * /64 first stage (factor 256) and nothing else queued, the mix is fused into the decimator kernel: a DEVICE capture is
 * then read in place (no staging copy) and, like hbd_push_samples_device, must stay valid and unchanged until the work
 * enqueued by the next hbd_process()/hbd_process_async() has passed it (work put on the handle's stream afterwards is
 * ordered behind that automatically).  hbd_push_samples_device with NCOs set is zero copy under the same conditions. */
int hbd_push_wideband(hbd_decoder* h, const float* iq, size_t n_complex, double sampling_rate);
int hbd_push_wideband_device(hbd_decoder* h, const float* d_iq, size_t n_complex, double sampling_rate);

/* ---- run (Decoder::process / operator(), Decoder.h:118-126,416-638) ------------------------------------- */
int hbd_process(hbd_decoder* h);        /* kernels + result drain + sentence layer + callbacks */
int hbd_process_async(hbd_decoder* h);  /* kernels only, returns immediately */
int hbd_collect(hbd_decoder* h);        /* drain results of all async calls so far (sentence layer + callbacks) */
/* like hbd_collect but leaves the newest `lag` calls in flight: the GPU keeps running while the host drains */
int hbd_collect_ready(hbd_decoder* h, unsigned lag);
/* Return channels to the state of channel 0 of a newly created handle with the same settings, e.g. to hand a channel of
 * a wideband receiver to a new payload (a new Decoder<float> in the reference).  Kept: the decimation plan, sampling
 * rate, FFT size, the handle-wide switches, and each channel's baud, framing, low-pass, dc_remove and NCO frequency.
 * Restarted: every filter history, the low-pass design, the spectrum and AFC, the slicer and UART, the demod
 * accumulation, SSDV and bit recording, the NCO phase (to 0), the text stream and last sentence, the SSDV image map.
 * Output not yet polled or gathered (characters, sentences, raw characters, SSDV packets) stays queued.
 * Every call in flight is drained first (callbacks fire before this returns, with the old text state); the reset itself
 * is one kernel on the handle's stream, ordered before the next call.  Out-of-range or duplicate channels: HBD_ERR_ARG;
 * samples pushed but not yet processed (in any channel): HBD_ERR_STATE; nothing is changed in either case.  n == 0: no-op.
 * The first call after a reset plans every channel on its own; from the second one on, batch and wideband pushes whose
 * size is a multiple of the factor are planned in O(1) of the channel count again (see hbd_get_kernel_timing, which 6). */
int hbd_reset_channels(hbd_decoder* h, const int* channels, size_t n);
int hbd_synchronize(hbd_decoder* h);
/* number of CUDA kernels this handle has launched so far */
unsigned long long hbd_kernel_launches(hbd_decoder* h);
/* measurement hook: on = 1 records CUDA events around every K1 (stage-1 decimator) launch, on = 2 also around the rest of
 * the step (two more event records per call on the low-priority stream); `which` 0 = K1, 1 = rest; 2..4 = signed pipeline gaps (K1 end -> next K1 start, K1 end -> own tail start,
 * tail end -> K1 start two calls later); 5 = host time of the drains' sentence-layer replay (count = calls drained);
 * 6 = host time of the calls' planning (count = frame counters stepped: one per FFT frame level in a call planned for all
 * channels at once, one per channel otherwise).
 * Calling set (on or off) clears the accumulated samples. */
int hbd_set_kernel_timing(hbd_decoder* h, int on);
int hbd_get_kernel_timing(hbd_decoder* h, int which, double* total_ms, unsigned* count);

/* ---- results ------------------------------------------------------------------------------------------ */
size_t hbd_get_rtty(hbd_decoder* h, int ch, char* out, size_t cap);           /* Decoder::getRTTY()         :642 */
size_t hbd_get_last_sentence(hbd_decoder* h, int ch, char* out, size_t cap);  /* Decoder::getLastSentence() :649 */
/* printable characters decoded since the previous poll == concat of character_callback_ payloads */
size_t hbd_poll_chars(hbd_decoder* h, int ch, char* out, size_t cap);
/* CRC-valid sentences since the previous poll, "callsign,data*crc\n" each == sentence_callback_ payloads */
size_t hbd_poll_sentences(hbd_decoder* h, int ch, char* out, size_t cap);
/* raw UART characters (what the reference hands to SSDV_wraper_t::push, Decoder.h:572-573) since the previous poll */
size_t hbd_poll_raw_chars(hbd_decoder* h, int ch, unsigned char* out, size_t cap);
/* retain raw characters for hbd_poll_raw_chars (default on; the reference itself keeps none, a caller that never polls
 * them switches it off) */
int    hbd_set_raw_chars(hbd_decoder* h, int on);
/* host threads hbd_collect* may use for the sentence layer of many channels (the caller's included); default min(4, half
 * the cores the process may run on).  Results and callback order do not depend on it. */
int    hbd_set_host_threads(hbd_decoder* h, int n);
int    hbd_set_sentence_callback(hbd_decoder* h, hbd_sentence_cb cb, void* user);
int    hbd_set_chars_callback(hbd_decoder* h, hbd_chars_cb cb, void* user);

/* ---- SSDV packet sync (the consumer of the raw characters: SSDV_wraper_t::push, code/Decoder/ssdv_wrapper.cpp:37-148,
 * fed once per process() that decoded characters, Decoder.h:572-573).  The 0x55 sync scan, the packet test
 * (CRC-32 + Reed-Solomon(255,223), the published algorithm of fsphil/ssdv's ssdv_dec_is_packet) and the per-image
 * packet bookkeeping (retransmitted id / changed resolution restart the image, :105-141) run here: the packet test on
 * the GPU for every channel, the bookkeeping on the host.  JPEG reassembly (ssdv_dec_feed, make_jpeg :151-172) is not
 * part of this library: hbd_get_ssdv_image returns exactly the packet sequence the reference feeds to it.
 * Off by default (nothing observable happens in the reference either until ssdv_callback_ is set, Decoder.h:141). */
typedef struct hbd_ssdv_packet_info {
    char callsign[8];      /* decoded base-40 callsign, NUL terminated (image key, ssdv_wrapper.cpp:105) */
    int  image_id, packet_id, width, height;
    int  errors;           /* symbols corrected by the Reed-Solomon decoder */
    int  set_size;         /* packets held for (callsign, image_id) now that this one is filed */
} hbd_ssdv_packet_info;
/* fires inside hbd_process()/hbd_collect*() once per accepted packet, like ssdv_callback_ (Decoder.h:631-632);
 * packet = the 256 corrected bytes */
typedef void (*hbd_ssdv_cb)(void* user, int ch, const hbd_ssdv_packet_info* info, const unsigned char* packet);
int    hbd_set_ssdv(hbd_decoder* h, int on);                               /* starts from an empty character stream */
int    hbd_set_ssdv_callback(hbd_decoder* h, hbd_ssdv_cb cb, void* user);  /* a non-NULL callback switches SSDV on */
/* accepted packets since the previous poll: infos[i], packets[256 * i]; returns the number available */
size_t hbd_poll_ssdv_packets(hbd_decoder* h, int ch, hbd_ssdv_packet_info* infos, unsigned char* packets, size_t cap_packets);
/* the packets filed under (callsign, image_id), 256 bytes each in packet-id order (input of make_jpeg); returns bytes */
size_t hbd_get_ssdv_image(hbd_decoder* h, int ch, const char* callsign, int image_id, unsigned char* out, size_t cap);
int    hbd_get_ssdv_last_image(hbd_decoder* h, int ch, char callsign[8], int* image_id);   /* last_img_k_, ssdv_wrapper.h:82 */
/* the packet test alone, batched on the GPU: windows[n][256] (host) are corrected in place where verdict[i] == 0
 * (packet) and left alone where verdict[i] == -1; errors[i] = corrected symbols */
int    hbd_ssdv_check_packets(hbd_decoder* h, unsigned char* windows, size_t n, int* verdict, int* errors);

/* ---- info (Decoder.h:98-101) ------------------------------------------------------------------------ */
int    hbd_get_decimation_factor(hbd_decoder* h);
double hbd_get_input_sampling_rate(hbd_decoder* h);
double hbd_get_decimated_sampling_rate(hbd_decoder* h);
double hbd_get_symbol_rate(hbd_decoder* h, int ch);
int    hbd_n_channels(hbd_decoder* h);

/* ---- GUI data (Decoder.h:104-115); sizes in floats, return = floats available -------------------------- */
size_t hbd_get_bins_count(hbd_decoder* h);
size_t hbd_get_fft(hbd_decoder* h, int ch, float* out_cf32, size_t cap_floats);
size_t hbd_get_demodulated(hbd_decoder* h, int ch, float* out, size_t cap_floats);
size_t hbd_get_power_spectrum(hbd_decoder* h, int ch, float* out, size_t cap_floats);
int    hbd_get_peaks(hbd_decoder* h, int ch, int* pl, int* pr);
int    hbd_get_noise_floor(hbd_decoder* h, int ch, double* nf, double* nv);
double hbd_get_shift(hbd_decoder* h, int ch);
double hbd_get_frequency_correction(hbd_decoder* h, int ch);
int    hbd_reset_frequency_correction(hbd_decoder* h, int ch, double frequency_correction);
size_t hbd_get_spectrum_info(hbd_decoder* h, int ch, hbd_spectrum_info* info, float* power, size_t cap_floats);
/* the per-channel record that is gathered to rank 0: out[6*ch + 0..5] = frequency correction, shift, noise floor,
 * noise variance, peak left, peak right (one device->host copy for all channels); returns 6*n_channels */
size_t hbd_get_stats_batch(hbd_decoder* h, double* out, size_t cap_doubles);

/* ---- multi-GPU result gather (SURVEY 8e) -------------------------------------------------------------------------
 * Channels are block-partitioned over ranks (one process per GPU, one hbd_decoder each) and never exchange signal data.
 * What travels, once per batch of calls, is one fixed-size record per channel with (the next piece of) what the reference's
 * callbacks and getters would have delivered since the previous gather: character_callback_ / sentence_callback_ payloads
 * (Decoder.h:135-138) and getFrequencyCorrection / getShift / getNoiseFloor / getPeaks (Decoder.h:108-113).
 * Rank 0 feeds the records into a host-only hbd_result_sink, which a server polls like a decoder.  The records can
 * travel over any transport (hbd_pack_results + hbd_sink_feed); hbd_dist_* / hbd_gather_results move them over NCCL
 * (bound at run time with dlopen: the library does not link against it). */
typedef struct hbd_result_record {          /* wire format, 256 bytes, little endian */
    uint32_t channel;                       /* global channel number */
    uint16_t n_chars;                       /* bytes used in chars[]: the next printable characters of the channel */
    uint16_t sentence_bytes;                /* bytes used in sentences[]: the next bytes of the channel's stream of CRC-valid
                                               sentences, "callsign,data*crc\n" each (a sentence may continue in the next record) */
    uint16_t n_sentences;                   /* '\n' terminators among them = sentences completed by this record */
    uint16_t flags;                         /* 1: more characters wait for the next record, 2: more sentence bytes wait */
    int32_t  peak_left, peak_right;
    float    frequency_correction, shift, noise_floor, noise_variance;
    uint32_t reserved;
    char     chars[88];
    char     sentences[128];
} hbd_result_record;
/* fill one record from the heads of a character stream and a sentence stream; *_used = bytes taken */
void   hbd_record_set(hbd_result_record* r, uint32_t channel, const char* chars, size_t n_chars, const char* sentences, size_t sentence_bytes,
                      const double stats[6], size_t* chars_used, size_t* sentence_bytes_used);
/* one record per local channel (channel = ch_offset + local index) with what hbd_poll_chars / hbd_poll_sentences would
 * return (and consumes it like they do) plus the AFC scalars as of the newest drained call; returns n_channels */
size_t hbd_pack_results(hbd_decoder* h, int ch_offset, hbd_result_record* out, size_t cap_records);
/* keep a per-call snapshot of the AFC scalars on the device so that hbd_pack_results never waits for calls in flight
 * (switched on by hbd_dist_init and by the first hbd_pack_results) */
int    hbd_set_stats_snapshot(hbd_decoder* h, int on);
typedef struct hbd_result_sink hbd_result_sink;
hbd_result_sink* hbd_sink_create(int total_channels);
void   hbd_sink_destroy(hbd_result_sink* s);
int    hbd_sink_feed(hbd_result_sink* s, const hbd_result_record* recs, size_t n);
int    hbd_sink_set_threads(hbd_result_sink* s, int n);   /* host threads a large feed may use (default min(4, cores)) */
size_t hbd_sink_poll_chars(hbd_result_sink* s, int ch, char* out, size_t cap);
size_t hbd_sink_poll_sentences(hbd_result_sink* s, int ch, char* out, size_t cap);
int    hbd_sink_stats(hbd_result_sink* s, int ch, double out[6]);   /* correction, shift, noise floor, noise variance, peak l, peak r */
void   hbd_sink_totals(hbd_result_sink* s, unsigned long long* chars, unsigned long long* sentences, unsigned long long* min_sentences,
                       unsigned long long* records);
/* a hash over every channel's character and sentence STREAMS (running CRC-32C per stream): independent of the sharding and of the gather cadence, so
 * the same channels decoded on 1, 2, 4 or 8 GPUs give the same value (the correctness check of SURVEY 8e) */
uint64_t hbd_sink_hash(hbd_result_sink* s);
/* NCCL transport.  Rank 0 draws an id (hbd_dist_unique_id) and hands the 128 bytes to the other ranks by any means; every
 * rank then calls hbd_dist_init (ncclCommInitRank on the handle's device), or adopts an ncclComm_t it already has. */
int    hbd_dist_unique_id(unsigned char out[128]);
int    hbd_dist_init(hbd_decoder* h, int rank, int world, const unsigned char id[128]);
int    hbd_dist_use_comm(hbd_decoder* h, void* nccl_comm, int rank, int world);
int    hbd_dist_finalize(hbd_decoder* h);
int    hbd_dist_total_channels(hbd_decoder* h);
/* every rank, at the same points of its call sequence: pack, ncclSend to rank 0 / ncclRecv there, feed `sink`: on rank 0
 * (required) with the records of ALL channels; on other ranks (optional, may be NULL) with the rank's own records, a local
 * mirror.  Global channel = channels of the lower ranks + local index.  Returns the records moved, < 0 on error.
 * Ranks > 0 only enqueue their send and return.  The sink takes the records in lazily (when it is polled, or a few gathers
 * later) and reads them from the handle's buffers until then: destroy a sink AFTER hbd_dist_finalize() / hbd_destroy() of
 * every handle that fed it. */
int    hbd_gather_results(hbd_decoder* h, hbd_result_sink* sink);

/* ---- websocket wire formats, produced on the GPU (the step after the path) -----------------------------------
 * PWR_ payload of "cmd::power:res=R,zoom=Z" (habdec_ws_protocol.cpp:353-404): SpectrumInfoHeader (NetTransport.h:29-47)
 * + the zoomed / shrunk dB spectrum as type_size-byte values (1: u8, 2: u16 min/max quantised like CompressedVector,
 * 4: f32).  Returns the payload size in bytes (0 before the first spectrum); copies min(cap, size). */
size_t hbd_get_spectrum_frame(hbd_decoder* h, int ch, float zoom, int resolution, int type_size, unsigned char* out, size_t cap);
/* all channels in one go: out[ch * pitch ...], sizes[ch]; returns the longest payload */
size_t hbd_get_spectrum_frames(hbd_decoder* h, float zoom, int resolution, int type_size, unsigned char* out, size_t pitch, unsigned* sizes);
/* DEM_ payload of "cmd::demod:res=R" (:408-429): DemodHeader + the accumulated discriminator output (last 50 symbols,
 * appended after every process() like websocketServer/main.cpp:267-282).  Accumulation is off until switched on. */
int    hbd_set_demod_accumulate(hbd_decoder* h, int on);
size_t hbd_get_demod_frame(hbd_decoder* h, int ch, int resolution, int type_size, unsigned char* out, size_t cap);
size_t hbd_get_demod_frames(hbd_decoder* h, int resolution, int type_size, unsigned char* out, size_t pitch, unsigned* sizes);

/* ---- telemetry layer (the consumer of the sentence callback: SentenceCallback, code/websocketServer/main.cpp:292-366).
 * Host only, no GPU involved: a few sentences per second and channel of scalar string work.  Three-way results follow
 * the reference: 1 = value, 0 = empty optional (too few fields, no GPS fix, unparsable time), -1 = the reference lets a
 * std::invalid_argument / out_of_range escape here (stoi / stof / string::at).  now_unix < 0 reads the system clock. */
enum { HBD_PARSE_OK = 1, HBD_PARSE_NONE = 0, HBD_PARSE_THROW = -1, HBD_PARSE_BADARG = -10 /* NULL pointer / malformed input */ };
typedef struct hbd_telemetry {          /* sondehub::MinTelemetry, code/sondehub/sondehub_uploader.h:12-21 */
    char  payload_callsign[64];         /* truncated to 63 characters */
    char  datetime[40];
    int   frame;
    float lat, lon, alt;
} hbd_telemetry;
typedef struct hbd_gps_distance {       /* habdec::GpsDistance, code/common/GpsDistance.h:7-14 */
    double dist_line_, dist_circle_, dist_radians_, elevation_, bearing_;
} hbd_gps_distance;
typedef struct hbd_channel_stats {      /* GLOBALS::STATS, code/websocketServer/GLOBALS.h:66-73 */
    unsigned num_ok_;
    hbd_gps_distance D_;
    double dist_max_, elev_min_;
    double age_s;                       /* seconds since last_sentence_timestamp_ */
} hbd_channel_stats;
int    hbd_parse_sentence(const char* sentence_without_crc, long long now_unix, hbd_telemetry* out);  /* sentence_parse.cpp:148-199 */
int    hbd_parse_sentence_time(const char* s, int* hour, int* minute, float* second);                 /* :50-68 */
int    hbd_parse_gps_pos(const char* s, float* out);                                                  /* :103-145 */
size_t hbd_timestamp_from_hms(int hour, int minute, float second, long long now_unix, char* out, size_t cap); /* :72-98 */
void   hbd_calc_gps_distance(double lat1, double lon1, double alt1, double lat2, double lon2, double alt2,
                             hbd_gps_distance* out);                                                  /* GpsDistance.cpp:21-84 */
/* "callsign,datetime,lat,lon,alt": what follows "cmd::info:tracking_telemetry=" (main.cpp:326-331) */
size_t hbd_tracking_telemetry_payload(const hbd_telemetry* t, char* out, size_t cap);
/* hbd_tracker: SentenceCallback + STATS + sentences_map_ for any number of channels (keys are caller-chosen channel
 * ids, e.g. global channel numbers on rank 0 after the gather).  Feed it by hand or attach it to a decoder handle. */
typedef struct hbd_tracker hbd_tracker;
typedef void (*hbd_telemetry_cb)(void* user, int ch, const hbd_telemetry* t, const char* sentence);
hbd_tracker* hbd_tracker_create(void);
void   hbd_tracker_destroy(hbd_tracker* t);
int    hbd_tracker_set_station(hbd_tracker* t, float lat, float lon, float alt);   /* PARAMS station_lat_/lon_/alt_ */
int    hbd_tracker_set_clock(hbd_tracker* t, long long now_unix);                  /* >= 0 freezes "today" (tests, replays) */
int    hbd_tracker_set_callback(hbd_tracker* t, hbd_telemetry_cb cb, void* user);
int    hbd_tracker_push(hbd_tracker* t, int ch, const char* callsign, const char* data, const char* crc);
int    hbd_tracker_push_sentence(hbd_tracker* t, int ch, const char* sentence);    /* "callsign,data*crc" as polled */
size_t hbd_tracker_poll(hbd_tracker* t, int ch, hbd_telemetry* out, size_t cap);   /* records since the previous poll */
/* channel `ch` as if no sentence had reached it: stats, sentences_map_ and unpolled records are dropped.  Pairs with
 * hbd_reset_channels when a channel is handed to a new payload (hbd_reset_channels leaves an attached tracker alone). */
int    hbd_tracker_reset(hbd_tracker* t, int ch);
int    hbd_tracker_stats(hbd_tracker* t, int ch, hbd_channel_stats* out);
/* "cmd::info:stats=ok:..,dist_line:..,...,alt:..[,age:..]" (habdec_ws_protocol.cpp:486-498) */
size_t hbd_tracker_stats_payload(hbd_tracker* t, int ch, int with_age, char* out, size_t cap);
size_t hbd_tracker_get_sentence(hbd_tracker* t, int ch, int frame, char* out, size_t cap);   /* sentences_map_[frame] */
/* every CRC-valid sentence of channel c is pushed to the tracker as channel c + ch_offset, on the processing thread,
 * after the sentence callback; NULL detaches */
int    hbd_attach_tracker(hbd_decoder* h, hbd_tracker* t, int ch_offset);

/* ---- wideband scanner (new; in the reference a person reads the spectrum and retunes the radio) ----------------
 * Finds 2-FSK (RTTY) payloads in a wideband capture and reports them as offsets from the capture centre, in the units
 * hbd_set_nco takes: hbd_set_nco(h, ch, sig.center_hz) puts a found signal at 0 Hz in channel ch.  Independent of
 * hbd_decoder; to scan the capture a decoder reads, give both the same stream and push the capture to both.
 *
 * Spectrum: N = n_fft (a power of two, 4096 .. 1048576), segments [s N/2, s N/2 + N) of the samples pushed since the last
 * reset (a segment is used once all its samples have arrived; samples wait across pushes), 4-term Blackman-Harris window
 * w (habdec_windows.h:27-53), P[k] = sum_s |X_s[k]|^2 / (S sum_n w[n]^2) with |X_s|^2 in float32 and the sum over
 * segments in float64, in segment order: the result does not depend on how the capture was cut into pushes.  Returned
 * fft-shifted as float32 (bin i = frequency (i - N/2) fs / N, the orientation of hbd_get_fft).  Integer formats are
 * dequantised exactly like a decoder push, so an integer push gives the PSD of the cf32 push of its dequantised values.
 * The first push latches fs; a push at another rate fails with HBD_ERR_STATE until hbd_scan_reset, which also clears
 * the spectrum and the waiting samples.  A device capture (16-byte aligned) is read in place by work enqueued on the
 * scanner's stream: it must stay valid and unchanged until that work has completed (work put on the stream later is
 * ordered behind it).  A host push returns when the caller owns `iq` again.  All entry points take the scanner's mutex.
 *
 * Detection (hbd_scan_find on the scanner's PSD, hbd_scan_detect on any PSD; host, float64): noise floor nf = lower
 * median of the 1024-bin block holding a bin; a tone candidate is a bin with P >= nf 10^(min_snr_db/10) that is the first
 * maximum of P within +-max(1, floor(min_shift_hz / (2 fs/N))) bins.  Strongest candidate first, each takes as partner
 * the strongest unused candidate between min_shift_hz and max_shift_hz away whose power is within max_tone_ratio_db of
 * its own; a pair uses up every candidate within one shift of it.  Detection is promised for baud <= shift only: faster
 * keying leaves no separate tones.  Signals come sorted by center_hz. */
typedef struct hbd_scanner hbd_scanner;
typedef struct hbd_scan_params {
    double min_snr_db, min_shift_hz, max_shift_hz, max_tone_ratio_db;   /* defaults 10, 150, 1200, 15 */
} hbd_scan_params;
typedef struct hbd_scan_signal {
    double center_hz, shift_hz, snr_db;   /* (f_a + f_b) / 2, |f_b - f_a|, 10 log10 min(P_a / nf_a, P_b / nf_b) */
    int    bin_lo, bin_hi;                /* the two tones' bins in the fft-shifted PSD */
} hbd_scan_signal;
int    hbd_scanner_create(int cuda_device, size_t n_fft, hbd_scanner** out);
void   hbd_scanner_destroy(hbd_scanner* s);
const char* hbd_scanner_last_error(hbd_scanner* s);
int    hbd_scanner_set_stream(hbd_scanner* s, void* cuda_stream);   /* share a decoder's stream to scan the same device capture */
int    hbd_scan_push(hbd_scanner* s, const void* iq, int format, size_t n_complex, double sampling_rate);
int    hbd_scan_push_device(hbd_scanner* s, const void* d_iq, int format, size_t n_complex, double sampling_rate);
int    hbd_scan_reset(hbd_scanner* s);
/* copies min(cap, N) floats of the PSD (zeros before the first complete segment); *n_segments = S; returns N */
size_t hbd_scan_get_psd(hbd_scanner* s, float* out, size_t cap_floats, unsigned long long* n_segments);
void   hbd_scan_default_params(hbd_scan_params* p);
/* signals found (may exceed cap; the first cap are stored), < 0 on error; p NULL = defaults */
int    hbd_scan_find(hbd_scanner* s, const hbd_scan_params* p, hbd_scan_signal* out, size_t cap);
int    hbd_scan_detect(const float* psd, size_t n, double fs, const hbd_scan_params* p, hbd_scan_signal* out, size_t cap);   /* host only */

/* ---- baud-rate estimation (new; in the reference a person types the rate into the web UI, cmd::set:baud) ----------
 * Measures each channel's keying rate on the GPU from its discriminator output d[i] (the floats hbd_debug_stage(
 * HBD_STAGE_DEMOD) returns, in stream order across calls; i counts samples since the estimator (re)started), so that a
 * channel tuned to a scanned signal can be set to its rate.  It only observes: no channel's decoding changes until the
 * caller applies a result.  Like the slicer it needs the tone pair to straddle DC (after the NCO).
 *
 * fs = fs_dec (hbd_get_decimated_sampling_rate); candidates B = {50, 75, 100, 150, 200, 300, 600} with fs / b >= 8;
 * debounce m = max(1, floor(fs / 2400)); histogram length Lmax = ceil(6.5 fs / 50).
 *  1. s[i] = d[i] > 0 (a zero counts as negative).
 *  2. The channel holds a current sign, taken from its first sample.  An edge is accepted once m consecutive samples have
 *     the opposite sign (a shorter opposite streak is discarded); its position is the first sample of that streak, and
 *     the current sign flips.
 *  3. For each accepted edge after the first, L = position - previous edge position: H[L] += 1 (uint32) if
 *     1 <= L <= Lmax, else long_runs += 1.  Streak and edge state carry across calls.
 *  4. On query, for each candidate b with sp = fs / b (double): a run L is explained by b when k = floor(L / sp + 0.5)
 *     has 1 <= k <= 6 and fabs(L - k sp) <= 0.2 sp (evaluated without fused multiply-adds).  E(b) = sum of H[L] over
 *     the explained runs (uint64).
 *  5. runs = sum H.  nominal = the lowest candidate with 10 E(b) >= 9 max E (integers: a harmonic explains the same runs,
 *     the lower rate wins); confidence = E(nominal) / runs; baud = fs * sum(H[L] k) / sum(H[L] L) over the runs nominal
 *     explains (uint64 sums, then double; 0 when it explains none): the payload's actual clock, e.g. 297.0 for a
 *     "300 baud" payload.  runs == 0: baud, nominal and confidence are 0.
 *
 * Off by default; while off it launches and allocates nothing.  On, it adds one kernel per call that does work, and
 * (Lmax + 1) * 4 bytes per channel (4 KB at fs_dec = 8 kHz, 40 KB at 78 125 Hz).  The estimator restarts (histograms and
 * edge state zeroed) when switched on, for the listed channels on hbd_reset_channels, and for every channel when the
 * decimation plan changes; the baud, framing, low-pass, NCO and FFT-size setters leave it alone.  Switching it on before
 * the first push sizes the rows at the first call.  A failed allocation returns HBD_ERR_NOMEM and changes nothing. */
typedef struct hbd_baud_estimate {
    double   baud;        /* fitted rate (step 5); 0: no run yet */
    double   nominal;     /* picked candidate of {50, 75, 100, 150, 200, 300, 600}; 0: no run yet */
    double   confidence;  /* E(nominal) / runs */
    unsigned runs;        /* runs histogrammed since the estimator (re)started */
    unsigned long_runs;   /* runs longer than the histogram (not in `runs`) */
} hbd_baud_estimate;
int    hbd_set_baud_estimation(hbd_decoder* h, int on);                         /* handle-wide, default off */
/* every channel, as of all calls enqueued so far (waits for them); out[0 .. min(cap, n_channels)); returns n_channels
 * (< 0: error; HBD_ERR_STATE when off) */
int    hbd_get_baud_estimates(hbd_decoder* h, hbd_baud_estimate* out, size_t cap);
/* where runs >= min_runs, confidence >= min_confidence and nominal != the channel's baud: exactly hbd_set_baud(h, ch,
 * nominal).  applied[n_channels] (may be NULL) receives the new rate or 0; returns the number of channels changed
 * (< 0: error; HBD_ERR_STATE when off) */
int    hbd_apply_baud_estimates(hbd_decoder* h, double min_confidence, unsigned min_runs, double* applied);
/* test hook: the channel's H[0 .. Lmax]; returns Lmax + 1 (0: bad channel, estimation off or no push yet) */
size_t hbd_get_baud_histogram(hbd_decoder* h, int ch, unsigned* out, size_t cap);

/* ---- test hooks ------------------------------------------------------------------------------------------ */
enum { HBD_STAGE_DECIMATED = 0, HBD_STAGE_FILTERED = 1, HBD_STAGE_DEMOD = 2, HBD_STAGE_LPTAPS = 5,
       HBD_STAGE_PENDING = 6, HBD_STAGE_BITS = 7 };
/* arrays of the most recent call (DECIMATED/FILTERED/DEMOD/BITS need hbd_set_record(h,1)); BITS accumulate */
size_t hbd_debug_stage(hbd_decoder* h, int ch, int stage, float* out, size_t cap_floats);
/* host half of the SSDV path alone (needs no GPU): the buffer automaton + bookkeeping replayed over n_chunks pushes
 * (chunk_sizes[i] characters each, empty chunks are skipped like calls without characters) with the accepted windows
 * given as (stream position, corrected packet, errors), ascending.  Returns the number of events; fills up to `cap`
 * of out_infos[i], out_chunk[i] (index of the push that filed the packet), out_packets[256 * i]. */
size_t hbd_ssdv_host_replay(const unsigned char* chars, const size_t* chunk_sizes, size_t n_chunks, const unsigned* accepted_pos,
                            const unsigned char* accepted_packets, const int* accepted_errors, size_t n_accepted,
                            hbd_ssdv_packet_info* out_infos, unsigned* out_chunk, unsigned char* out_packets, size_t cap);
/* low-pass tap design alone (FirFilter::LP_BlackmanHarris, FirFilter.h:173-209); returns the tap count */
size_t hbd_design_lowpass(float rel_width, float trans, size_t input_size, size_t current_taps, float* out, size_t cap);
/* sentence layer alone (extractSentence + CRC, sentence_extract.cpp:58-98, CRC.cpp:21-47):
 * returns 1 and fills the fields if a sentence was found; *rest_offset = start of the remaining stream */
int    hbd_extract_sentence(const char* stream, size_t n, char* callsign, char* data, char* crc, size_t cap, size_t* rest_offset);
void   hbd_crc16(const char* s, size_t n, char out[5]);
/* the text layer alone (printable filter + sentence scan + trims, Decoder.h:572-613,635-636; needs no GPU): n_chunks pushes of
 * raw characters; out = "<CRC-valid sentences, one per line>\x1e<last sentence>\x1e<text stream>"; returns its size */
size_t hbd_text_replay(const unsigned char* chars, const size_t* chunk_sizes, size_t n_chunks, char* out, size_t cap);

#ifdef __cplusplus
}
#endif
#endif
