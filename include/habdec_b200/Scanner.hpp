// C++17 facade over the wideband scanner of the C ABI (include/habdec_b200.h, hbd_scanner / hbd_scan_*): an averaged
// GPU spectrum of a capture and the RTTY tone pairs in it, as offsets from the capture centre that BatchDecoder::nco takes.
//
//   habdec_b200::Scanner scan(1 << 20);
//   scan.push(capture);                                  // or pushDevice(ptr, format, n, fs) on the decoder's stream
//   for (const hbd_scan_signal& s : scan.find()) dec.nco(s.center_hz, free_channel());
//
// Header only; link with -lhabdec_b200.
#pragma once
#include <stdexcept>
#include <string>
#include <vector>

#include "../habdec_b200.h"
#include "Decoder.hpp"

namespace habdec_b200 {

class Scanner {
public:
    explicit Scanner(size_t n_fft, int cuda_device = 0) : n_(n_fft)
    {
        const int rc = hbd_scanner_create(cuda_device, n_fft, &s_);
        if (rc == HBD_ERR_ARG) throw std::invalid_argument("habdec_b200::Scanner: n_fft must be a power of two in [4096, 2^20]");
        if (rc != HBD_OK) throw std::runtime_error("habdec_b200::Scanner: no usable CUDA device (there is no CPU fallback)");
    }
    ~Scanner() { hbd_scanner_destroy(s_); }
    Scanner(const Scanner&) = delete;
    Scanner& operator=(const Scanner&) = delete;

    hbd_scanner* handle() { return s_; }
    size_t size() const { return n_; }
    const char* lastError() { return hbd_scanner_last_error(s_); }
    bool setStream(void* cuda_stream) { return hbd_scanner_set_stream(s_, cuda_stream) == HBD_OK; }

    // host captures: cf32 (rate from the IQVector) or integer IQ; device captures are read in place on the scanner's stream
    bool push(const IQVector& v) { return hbd_scan_push(s_, v.data(), HBD_IQ_CF32, v.size(), v.samplingRate()) == HBD_OK; }
    bool push(const void* iq, hbd_iq_format format, size_t n, double fs) { return hbd_scan_push(s_, iq, format, n, fs) == HBD_OK; }
    bool pushDevice(const void* d_iq, size_t n, double fs) { return hbd_scan_push_device(s_, d_iq, HBD_IQ_CF32, n, fs) == HBD_OK; }
    bool pushDevice(const void* d_iq, hbd_iq_format format, size_t n, double fs) { return hbd_scan_push_device(s_, d_iq, format, n, fs) == HBD_OK; }
    bool reset() { return hbd_scan_reset(s_) == HBD_OK; }

    // fft-shifted PSD (bin i: (i - N/2) fs / N), empty on error; segments averaged into it
    std::vector<float> psd(unsigned long long* n_segments = nullptr)
    {
        std::vector<float> out(n_);
        if (hbd_scan_get_psd(s_, out.data(), out.size(), n_segments) != n_) out.clear();
        return out;
    }

    static hbd_scan_params defaultParams()
    {
        hbd_scan_params p;
        hbd_scan_default_params(&p);
        return p;
    }

    // signals sorted by center_hz; throws on error
    std::vector<hbd_scan_signal> find(const hbd_scan_params& p = defaultParams())
    {
        std::vector<hbd_scan_signal> out(16);
        int n = hbd_scan_find(s_, &p, out.data(), out.size());
        if (n > int(out.size())) {
            out.resize(size_t(n));
            n = hbd_scan_find(s_, &p, out.data(), out.size());
        }
        if (n < 0) throw std::runtime_error(std::string("habdec_b200::Scanner::find: ") + lastError());
        out.resize(size_t(n));
        return out;
    }

private:
    size_t n_;
    hbd_scanner* s_ = nullptr;
};

} // namespace habdec_b200
