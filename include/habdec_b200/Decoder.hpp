// C++17 facade over the C ABI (include/habdec_b200.h) with the reference's member names, so that code written
// against habdec::Decoder<float> (code/Decoder/Decoder.h:65-141) -- e.g. DECODER_THREAD in
// code/websocketServer/main.cpp:203-283 -- compiles against the B200 implementation by changing one type.
//
//   habdec_b200::Decoder        one channel  == one reference Decoder<float>
//   habdec_b200::BatchDecoder   N channels processed together (the reason this library exists)
//
// Header only; link with -lhabdec_b200.
#pragma once
#include <algorithm>
#include <complex>
#include <cstdint>
#include <cstdlib>
#include <functional>
#include <stdexcept>
#include <string>
#include <vector>

#include "../habdec_b200.h"

namespace habdec_b200 {

// same shape as habdec::IQVector<float> (code/Decoder/IQVector.h:33-64): a complex vector that knows its rate
class IQVector : public std::vector<std::complex<float>> {
public:
    double samplingRate() const { return sampling_rate_; }
    void samplingRate(double r) { sampling_rate_ = r; }
private:
    double sampling_rate_ = 0;
};

// same shape as habdec::SpectrumInfo<T> (code/Decoder/SpectrumInfo.h:35-85): the dB power spectrum as a vector with the
// AFC's findings attached; callers erase / shrink it in place (habdec_ws_protocol.cpp:355-405)
template <typename T>
class SpectrumInfo : public std::vector<T> {
public:
    typedef T TValue;
    mutable T min_ = 0;
    mutable T max_ = 0;
    mutable double noise_floor_ = 0;
    mutable double noise_variance_ = 0;
    mutable double sampling_rate_ = 0;
    mutable double shift_ = 0;
    mutable int peak_left_ = 0;
    mutable int peak_right_ = 0;
    mutable bool peak_left_valid_ = false;
    mutable bool peak_right_valid_ = false;

    SpectrumInfo() = default;
    template <typename U>
    SpectrumInfo(const SpectrumInfo<U>& rhs)   // like the reference's, min/max, rate and shift are not carried over
        : std::vector<T>(rhs.begin(), rhs.end()), noise_floor_(rhs.noise_floor_), noise_variance_(rhs.noise_variance_), peak_left_(rhs.peak_left_),
          peak_right_(rhs.peak_right_), peak_left_valid_(rhs.peak_left_valid_), peak_right_valid_(rhs.peak_right_valid_) {}
    template <typename U>
    const SpectrumInfo<T>& operator=(const SpectrumInfo<U>& rhs)
    {
        std::vector<T>::assign(rhs.begin(), rhs.end());
        noise_floor_ = rhs.noise_floor_; noise_variance_ = rhs.noise_variance_;
        peak_left_ = rhs.peak_left_; peak_right_ = rhs.peak_right_;
        peak_left_valid_ = rhs.peak_left_valid_; peak_right_valid_ = rhs.peak_right_valid_;
        return *this;
    }
    const SpectrumInfo<T>& operator=(const std::vector<T>& rhs) { std::vector<T>::operator=(rhs); return *this; }
};

class BatchDecoder {
public:
    explicit BatchDecoder(int n_channels, int cuda_device = 0)
    {
        if (hbd_create(n_channels, cuda_device, &h_) != HBD_OK)
            throw std::runtime_error("habdec_b200: no usable CUDA device (there is no CPU fallback)");
    }
    ~BatchDecoder() { hbd_destroy(h_); }
    BatchDecoder(const BatchDecoder&) = delete;
    BatchDecoder& operator=(const BatchDecoder&) = delete;

    int channels() const { return hbd_n_channels(h_); }
    hbd_decoder* handle() { return h_; }

    // feed: one channel, all channels from a host matrix, or a device matrix (zero copy)
    bool pushSamples(int ch, const IQVector& v) { return hbd_push_samples(h_, ch, reinterpret_cast<const float*>(v.data()), v.size(), v.samplingRate()) == HBD_OK; }
    bool pushSamples(const std::complex<float>* host_matrix, size_t n, size_t pitch, double fs) { return hbd_push_samples_batch(h_, reinterpret_cast<const float*>(host_matrix), n, pitch, fs) == HBD_OK; }
    bool pushSamplesDevice(const void* device_matrix, size_t n, size_t pitch, double fs) { return hbd_push_samples_device(h_, static_cast<const float*>(device_matrix), n, pitch, fs) == HBD_OK; }
    // the same from integer IQ (CS16 / CS8 / CU8 as receivers deliver it; n, pitch in complex samples)
    bool pushSamples(int ch, const void* iq, hbd_iq_format format, size_t n, double fs) { return hbd_push_iq(h_, ch, iq, format, n, fs) == HBD_OK; }
    bool pushSamples(const void* host_matrix, hbd_iq_format format, size_t n, size_t pitch, double fs) { return hbd_push_iq_batch(h_, host_matrix, format, n, pitch, fs) == HBD_OK; }
    bool pushSamplesDevice(const void* device_matrix, hbd_iq_format format, size_t n, size_t pitch, double fs) { return hbd_push_iq_device(h_, device_matrix, format, n, pitch, fs) == HBD_OK; }

    // one wideband capture for all channels, each through its own NCO (frequency-offset channels)
    bool pushWideband(const IQVector& v) { return hbd_push_wideband(h_, reinterpret_cast<const float*>(v.data()), v.size(), v.samplingRate()) == HBD_OK; }
    bool pushWidebandDevice(const void* device_row, size_t n, double fs) { return hbd_push_wideband_device(h_, static_cast<const float*>(device_row), n, fs) == HBD_OK; }
    bool pushWideband(const void* row, hbd_iq_format format, size_t n, double fs) { return hbd_push_iq_wideband(h_, row, format, n, fs) == HBD_OK; }
    bool pushWidebandDevice(const void* device_row, hbd_iq_format format, size_t n, double fs) { return hbd_push_iq_wideband_device(h_, device_row, format, n, fs) == HBD_OK; }
    // NCO pre-mixer: replaces the SDR retune of code/websocketServer/main.cpp:247-265
    void nco(double freq_hz, int ch = -1) { hbd_set_nco(h_, ch, freq_hz); }
    double nco(int ch) const { return hbd_get_nco(h_, ch); }
    int afcRetune(double min_abs_hz = 100.0, double* applied = nullptr) { return hbd_afc_retune(h_, min_abs_hz, applied); }
    // baud-rate estimation (include/habdec_b200.h): every channel's keying rate measured on the GPU, applied on request
    int setBaudEstimation(bool on) { return status_ = hbd_set_baud_estimation(h_, on ? 1 : 0); }
    std::vector<hbd_baud_estimate> getBaudEstimates()
    {
        std::vector<hbd_baud_estimate> v(static_cast<size_t>(channels()));
        status_ = hbd_get_baud_estimates(h_, v.data(), v.size());
        if (status_ < 0) v.clear(); else status_ = HBD_OK;
        return v;
    }
    // returns the number of channels retuned (< 0: error); applied[channels()] may be null
    int applyBaudEstimates(double min_confidence = 0.8, unsigned min_runs = 100, double* applied = nullptr)
    {
        const int rc = hbd_apply_baud_estimates(h_, min_confidence, min_runs, applied);
        status_ = rc < 0 ? rc : HBD_OK;
        return rc;
    }

    // configure (ch = -1: every channel)
    void baud(double v, int ch = -1) { hbd_set_baud(h_, ch, v); }
    double baud(int ch) const { return hbd_get_baud(h_, ch); }
    void rtty_bits(size_t v, int ch = -1) { hbd_set_rtty_bits(h_, ch, v); }
    size_t rtty_bits(int ch) const { return hbd_get_rtty_bits(h_, ch); }
    void rtty_stops(float v, int ch = -1) { hbd_set_rtty_stops(h_, ch, v); }
    float rtty_stops(int ch) const { return hbd_get_rtty_stops(h_, ch); }
    void lowpass_bw(float v, int ch = -1) { hbd_set_lowpass_bw(h_, ch, v); }
    float lowpass_bw(int ch) const { return hbd_get_lowpass_bw(h_, ch); }
    void lowpass_trans(float v, int ch = -1) { hbd_set_lowpass_trans(h_, ch, v); }
    float lowpass_trans(int ch) const { return hbd_get_lowpass_trans(h_, ch); }
    void dc_remove(bool v, int ch = -1) { hbd_set_dc_remove(h_, ch, v); }
    bool dc_remove(int ch) const { return hbd_get_dc_remove(h_, ch) != 0; }
    size_t setupDecimationStagesFactor(size_t f) { return hbd_setup_decimation_factor(h_, f); }
    size_t setupDecimationStagesBW(double max_rate) { return hbd_setup_decimation_bw(h_, max_rate); }

    // run.  The reference's process() returns nothing and reports trouble on stdout; here the status of the last call is
    // kept (lastStatus() / lastError()) and returned by the int-returning forms.
    int process() { return status_ = hbd_process(h_); }
    void operator()() { process(); }
    int processAsync() { return status_ = hbd_process_async(h_); }
    int collect() { return status_ = hbd_collect(h_); }
    int collectReady(unsigned lag) { return status_ = hbd_collect_ready(h_, lag); }
    // channels start over like a new Decoder<float> with the same settings (hbd_reset_channels); unpolled output stays queued
    int resetChannels(const std::vector<int>& chs) { return status_ = hbd_reset_channels(h_, chs.data(), chs.size()); }
    int resetChannel(int ch) { return resetChannels({ch}); }
    int lastStatus() const { return status_; }
    std::string lastError() const { return hbd_last_error(h_); }

    // results
    std::string getRTTY(int ch) { return str(hbd_get_rtty, ch); }
    std::string getLastSentence(int ch) { return str(hbd_get_last_sentence, ch); }
    std::string pollChars(int ch) { return str(hbd_poll_chars, ch); }
    std::string pollSentences(int ch) { return str(hbd_poll_sentences, ch); }

    // info
    int getDecimationFactor() const { return hbd_get_decimation_factor(h_); }
    double getInputSamplingRate() const { return hbd_get_input_sampling_rate(h_); }
    double getDecimatedSamplingRate() const { return hbd_get_decimated_sampling_rate(h_); }
    double getSymbolRate(int ch) const { return hbd_get_symbol_rate(h_, ch); }

    // GUI data
    size_t getBinsCount() const { return hbd_get_bins_count(h_); }
    IQVector getFFT(int ch)
    {
        IQVector v; v.resize(hbd_get_fft(h_, ch, nullptr, 0) / 2);
        if (!v.empty()) hbd_get_fft(h_, ch, reinterpret_cast<float*>(v.data()), 2 * v.size());
        v.samplingRate(getDecimatedSamplingRate());
        return v;
    }
    std::vector<float> getDemodulated(int ch) { return floats(hbd_get_demodulated, ch); }
    std::vector<float> getPowerSpectrum(int ch) { return floats(hbd_get_power_spectrum, ch); }
    void getPeaks(int ch, int& pl, int& pr) { hbd_get_peaks(h_, ch, &pl, &pr); }
    void getNoiseFloor(int ch, double& nf, double& nv) { hbd_get_noise_floor(h_, ch, &nf, &nv); }
    double getShift(int ch) { return hbd_get_shift(h_, ch); }
    double getFrequencyCorrection(int ch) { return hbd_get_frequency_correction(h_, ch); }
    void resetFrequencyCorrection(int ch, double c) { hbd_reset_frequency_correction(h_, ch, c); }
    // Decoder::getSpectrumInfo (Decoder.h:115,814-836)
    SpectrumInfo<float> getSpectrumInfo(int ch)
    {
        SpectrumInfo<float> si;
        hbd_spectrum_info info;
        si.resize(getBinsCount());
        const size_t n = hbd_get_spectrum_info(h_, ch, &info, si.data(), si.size());
        si.resize(std::min(n, si.size()));
        if (si.empty()) return si;                       // no spectrum yet: an empty vector with default fields (:818-819)
        si.min_ = info.min_; si.max_ = info.max_;
        si.noise_floor_ = info.noise_floor_; si.noise_variance_ = info.noise_variance_;
        si.sampling_rate_ = info.sampling_rate_; si.shift_ = info.shift_;
        si.peak_left_ = info.peak_left_; si.peak_right_ = info.peak_right_;
        si.peak_left_valid_ = info.peak_left_valid_ != 0; si.peak_right_valid_ = info.peak_right_valid_ != 0;
        return si;
    }

    // SSDV (Decoder.h:141,572-573,631-632): switched on by installing ssdv_callback_ (or ssdv(true)); packets are polled or
    // delivered through the callback
    void ssdv(bool on) { hbd_set_ssdv(h_, on ? 1 : 0); }
    std::vector<uint8_t> getSsdvImagePackets(int ch, const std::string& callsign, int image_id)
    {
        std::vector<uint8_t> v(hbd_get_ssdv_image(h_, ch, callsign.c_str(), image_id, nullptr, 0));
        if (!v.empty()) hbd_get_ssdv_image(h_, ch, callsign.c_str(), image_id, v.data(), v.size());
        return v;
    }

    // callbacks: (channel, callsign, data, crc) / (channel, chars) / (channel, callsign, image id, bytes); fired by
    // process()/collect() on the calling thread, after the handle's lock is released (they may call back into the decoder)
    std::function<void(int, std::string, std::string, std::string)> sentence_callback_;
    std::function<void(int, std::string)> character_callback_;
    // like Decoder::ssdv_callback_(callsign, image_id, jpeg).  The bytes are what ssdv_jpeg_ makes of the image's packets
    // (256 bytes each, packet-id order: exactly what the reference feeds to ssdv_dec_feed, ssdv_wrapper.cpp:151-172); JPEG
    // reassembly lives in fsphil/ssdv, which is not part of this library -- link it and set ssdv_jpeg_ to a function that
    // runs ssdv_dec_feed / ssdv_dec_get_jpeg over the packets.  Without it the packets themselves are handed over.
    std::function<void(int, std::string, int, std::vector<uint8_t>)> ssdv_callback_;
    std::function<std::vector<uint8_t>(const std::vector<uint8_t>& packets)> ssdv_jpeg_;
    void installCallbacks()
    {
        hbd_set_sentence_callback(h_, sentence_callback_ ? &BatchDecoder::on_sentence : nullptr, this);
        hbd_set_chars_callback(h_, character_callback_ ? &BatchDecoder::on_chars : nullptr, this);
        if (ssdv_callback_) hbd_set_ssdv_callback(h_, &BatchDecoder::on_ssdv, this);
    }

private:
    static void on_sentence(void* u, int ch, const char* cs, const char* d, const char* crc) { static_cast<BatchDecoder*>(u)->sentence_callback_(ch, cs, d, crc); }
    static void on_chars(void* u, int ch, const char* p, size_t n) { static_cast<BatchDecoder*>(u)->character_callback_(ch, std::string(p, n)); }
    static void on_ssdv(void* u, int ch, const hbd_ssdv_packet_info* info, const unsigned char*)
    {
        BatchDecoder* self = static_cast<BatchDecoder*>(u);
        if (!self->ssdv_callback_) return;
        std::vector<uint8_t> bytes = self->getSsdvImagePackets(ch, info->callsign, info->image_id);   // get_jpeg(last_img_k_), Decoder.h:632
        if (self->ssdv_jpeg_) bytes = self->ssdv_jpeg_(bytes);
        self->ssdv_callback_(ch, info->callsign, info->image_id, std::move(bytes));
    }
    template <typename F> std::string str(F fn, int ch)
    {
        std::string s(fn(h_, ch, nullptr, 0), '\0');
        if (!s.empty()) fn(h_, ch, &s[0], s.size());
        return s;
    }
    template <typename F> std::vector<float> floats(F fn, int ch)
    {
        std::vector<float> v(fn(h_, ch, nullptr, 0));
        if (!v.empty()) fn(h_, ch, v.data(), v.size());
        return v;
    }
    hbd_decoder* h_ = nullptr;
    int status_ = HBD_OK;
};

// One channel with the reference's public surface (Decoder.h:73-141): every public member of habdec::Decoder<float> has its
// counterpart here, so DECODER_THREAD (websocketServer/main.cpp:203-283), the callback installs (:573-604) and
// SpectrumToStream (habdec_ws_protocol.cpp:355-405) compile against it (tests/cpp/decoder_thread.cpp).  livePrint /
// ssdvBaseFile are kept as inert properties: the text console and the JPEG file writer are outside the accelerated path.
class Decoder {
public:
    explicit Decoder(int cuda_device = 0) : b_(1, cuda_device) {}
    bool pushSamples(const IQVector& v) { return b_.pushSamples(0, v); }
    bool pushSamples(const void* iq, hbd_iq_format format, size_t n, double fs) { return b_.pushSamples(0, iq, format, n, fs); }   // integer IQ
    void lowpass_bw(float v) { b_.lowpass_bw(v, 0); }
    float lowpass_bw() const { return b_.lowpass_bw(0); }
    void lowpass_trans(float v) { b_.lowpass_trans(v, 0); }
    float lowpass_trans() const { return b_.lowpass_trans(0); }
    void baud(double v) { b_.baud(v, 0); }
    double baud() const { return b_.baud(0); }
    void rtty_bits(size_t v) { b_.rtty_bits(v, 0); }
    size_t rtty_bits() const { return b_.rtty_bits(0); }
    void rtty_stops(float v) { b_.rtty_stops(v, 0); }
    float rtty_stops() const { return b_.rtty_stops(0); }
    void dc_remove(bool v) { b_.dc_remove(v, 0); }
    bool dc_remove() const { return b_.dc_remove(0); }
    size_t setupDecimationStagesFactor(size_t f) { return b_.setupDecimationStagesFactor(f); }
    size_t setupDecimationStagesBW(double r) { return b_.setupDecimationStagesBW(r); }
    std::string getRTTY() { return b_.getRTTY(0); }
    std::string getLastSentence() { return b_.getLastSentence(0); }
    int getDecimationFactor() const { return b_.getDecimationFactor(); }
    double getInputSamplingRate() const { return b_.getInputSamplingRate(); }
    double getDecimatedSamplingRate() const { return b_.getDecimatedSamplingRate(); }
    double getSymbolRate() const { return b_.getSymbolRate(0); }
    size_t getBinsCount() const { return b_.getBinsCount(); }
    IQVector getFFT() { return b_.getFFT(0); }
    std::vector<float> getDemodulated() { return b_.getDemodulated(0); }
    std::vector<float> getPowerSpectrum() { return b_.getPowerSpectrum(0); }
    void getPeaks(int& pl, int& pr) { b_.getPeaks(0, pl, pr); }
    void getNoiseFloor(double& nf, double& nv) { b_.getNoiseFloor(0, nf, nv); }
    double getShift() { return b_.getShift(0); }
    double getFrequencyCorrection() { return b_.getFrequencyCorrection(0); }
    void resetFrequencyCorrection(double c) { b_.resetFrequencyCorrection(0, c); }
    SpectrumInfo<float> getSpectrumInfo() { return b_.getSpectrumInfo(0); }
    void process()
    {
        if (!wired_ || (ssdv_callback_ && !ssdv_wired_)) {
            b_.sentence_callback_ = [this](int, std::string a, std::string b, std::string c) { if (sentence_callback_) sentence_callback_(a, b, c); };
            b_.character_callback_ = [this](int, std::string s) { if (character_callback_) character_callback_(s); };
            if (ssdv_callback_) {
                b_.ssdv_jpeg_ = ssdv_jpeg_;
                b_.ssdv_callback_ = [this](int, std::string cs, int id, std::vector<uint8_t> bytes) { if (ssdv_callback_) ssdv_callback_(cs, id, std::move(bytes)); };
                ssdv_wired_ = true;
            }
            b_.installCallbacks();
            wired_ = true;
        }
        b_.process();
    }
    void operator()() { process(); }
    int lastStatus() const { return b_.lastStatus(); }
    std::string lastError() const { return b_.lastError(); }
    BatchDecoder& batch() { return b_; }                 // the one-channel batch behind this decoder (C ABI handle: batch().handle())
    bool livePrint() const { return live_print_; }
    void livePrint(bool v) { live_print_ = v; }
    std::string ssdvBaseFile() const { return ssdv_base_; }
    void ssdvBaseFile(const std::string& f) { ssdv_base_ = f; }
    std::function<void(std::string, std::string, std::string)> sentence_callback_;   // Decoder.h:135
    std::function<void(std::string)> character_callback_;                            // Decoder.h:138
    std::function<void(std::string, int, std::vector<uint8_t>)> ssdv_callback_;      // Decoder.h:141 (see BatchDecoder::ssdv_callback_ for the bytes)
    std::function<std::vector<uint8_t>(const std::vector<uint8_t>& packets)> ssdv_jpeg_;
private:
    BatchDecoder b_;
    bool wired_ = false, ssdv_wired_ = false, live_print_ = false;
    std::string ssdv_base_;
};

} // namespace habdec_b200
